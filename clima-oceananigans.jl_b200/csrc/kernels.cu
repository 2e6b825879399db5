// kernels.cu -- halo fills, general tendency(+substep), pressure rhs / correction, hydrostatic
// pressure, layout conversion and reductions.  sm_100a.
#include "internal.h"
#include <algorithm>
#include <cstdlib>

namespace ob {

// =============================================================================================
// fill_halo_regions!  (BoundaryConditions/fill_halo_regions*.jl)
// One launch per dimension for ALL fields of the batch.  Periodic dims copy H planes over the
// full allocated extent of the other two dims (fills edges/corners when applied dim after dim);
// Bounded dims act on the interior extent of the other dims only, first halo cell only.
// =============================================================================================
template <class FT>
__global__ void fill_halo_kernel(GridD<FT> g, HaloBatch<FT> hb, int d, int a, int b, int alo, int ahi,
                                 int blo, int bhi) {
    int ia = alo + blockIdx.x * blockDim.x + threadIdx.x;
    int ib = blo + blockIdx.y * blockDim.y + threadIdx.y;
    if (ia > ahi || ib > bhi) return;
    long long base = ia * g.st[a] + ib * g.st[b];
    long long s = g.st[d];
    int N = g.N[d], H = g.H[d];
    if (g.topo[d] == OB_PERIODIC) {
        for (int n = 0; n < hb.n; ++n) {
            FT* f = hb.p0[n] + base;
            for (int h = 1; h <= H; ++h) {
                f[(h - H) * s] = f[(N + h - H) * s];        // c[i] = c[N+i], i = 1-H..0
                f[(N + h) * s] = f[h * s];                  // c[N+i] = c[i], i = 1..H
            }
        }
    } else if (g.topo[d] == OB_BOUNDED) {
        for (int n = 0; n < hb.n; ++n) {
            FT* f = hb.p0[n] + base;
            for (int side = 0; side < 2; ++side) {
                int kind = hb.bc_kind[n][2 * d + side];
                // getbc(bc::BC{<:Any,<:AbstractArray}, i, j, grid) = bc.condition[i, j] (boundary_condition.jl): the array
                // spans the interior extent (1..ahi) x (1..bhi) of the tangential dimensions, alo = blo = 1 here
                const FT* tab = hb.bc_tab[n][2 * d + side];
                FT val = tab ? tab[(ia - 1) + (long long)(ib - 1) * ahi] : hb.bc_val[n][2 * d + side];
                if (kind == 2) {                            // Flux: mirror (fill_halo_regions_flux.jl:16-28)
                    if (side == 0) f[0] = f[s];
                    else f[(N + 1) * s] = f[N * s];
                } else if (kind == 5) {                     // Open (fill_halo_regions_open.jl:34-39)
                    f[(side == 0 ? 1 : N + 1) * s] = val;
                } else if (kind == 3 || kind == 4) {        // Value / Gradient (…_value_gradient.jl:7-99)
                    int iB = side == 0 ? 1 : N + 1, iI = side == 0 ? 1 : N, iH = side == 0 ? 0 : N + 1;
                    FT D = spacing(g, d, hb.loc[n][d] == OB_C ? OB_F : OB_C, iB);
                    FT cI = f[iI * s];
                    FT grad = kind == 4 ? val : (side == 0 ? (cI - val) / (D / 2) : (val - cI) / (D / 2));
                    f[iH * s] = cI + grad * (side == 0 ? -D : D);
                }
            }
        }
    }
}

// ---- all non-Flat dimensions Periodic (or slab-decomposed): ONE launch for all dimensions and all fields --------
// Applying the periodic copies x, then y, then z (fill_halo_regions_periodic.jl:15-105) gives every halo cell --
// edges and corners included -- the value of the interior cell obtained by wrapping each of its indices.  The
// shell kernel writes exactly that, reading cells that no thread of the launch writes, so there is no ordering
// between dimensions.  The shell is enumerated as up to three groups, one per Periodic dimension D (z, y, x in
// that order): index along D in the 2H halo planes; the dimensions enumerated before D over their interior (their
// halo cells belong to the earlier group), the others over their full extent.  A slab-decomposed (FullyConnected)
// dimension has no group of its own -- its halos come from the neighbour exchange, done BEFORE this launch on the
// interior extent of the other dimensions -- but it is always walked over its full extent and never wrapped, so
// the corner cells pick up the exchanged values.
struct ShellGroup { int D, HD, lo[3], n[3]; long long count; };    // HD: a FullyConnected dimension walked over its 2H halo rows only (-1: none)
struct ShellPlan { ShellGroup g[3]; int ng; long long total; };

template <class FT>
__global__ void __launch_bounds__(256) fill_halo_shell_kernel(GridD<FT> g, HaloBatch<FT> hb, ShellPlan P) {
    long long t = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    if (t >= P.total) return;
    int q = 0;
    while (q + 1 < P.ng && t >= P.g[q].count) { t -= P.g[q].count; ++q; }
    const ShellGroup& G = P.g[q];
    int id[3];
    {   // x fastest
        long long r = t / G.n[0];
        id[0] = (int)(t - r * G.n[0]);
        long long r2 = r / G.n[1];
        id[1] = (int)(r - r2 * G.n[1]);
        id[2] = (int)r2;
    }
    long long dst = 0, src = 0;
#pragma unroll
    for (int d = 0; d < 3; ++d) {
        int v;
        if (d == G.D || d == G.HD) v = id[d] < g.H[d] ? id[d] + 1 - g.H[d] : g.N[d] + 1 + (id[d] - g.H[d]);
        else v = G.lo[d] + id[d];
        int sv = v;
        if (g.topo[d] == OB_PERIODIC) sv = v < 1 ? v + g.N[d] : (v > g.N[d] ? v - g.N[d] : v);
        dst += v * g.st[d];
        src += sv * g.st[d];
    }
    FT v[MAXF];
#pragma unroll
    for (int n = 0; n < MAXF; ++n) if (n < hb.n) v[n] = hb.p0[n][src];
#pragma unroll
    for (int n = 0; n < MAXF; ++n) if (n < hb.n) hb.p0[n][dst] = v[n];
}
// `with_comm`: a FullyConnected dimension is allowed (the caller exchanges it first)
template <class FT>
static bool shell_fill_supported(const GridD<FT>& g, bool with_comm) {
    bool any = false;
    for (int d = 0; d < 3; ++d) {
        if (g.topo[d] == OB_FLAT) continue;
        if (g.topo[d] == OB_COMM) { if (!with_comm) return false; continue; }
        if (g.topo[d] != OB_PERIODIC || g.H[d] < 1 || g.N[d] < g.H[d]) return false;
        any = true;
    }
    return any;
}
// comm_rows: how a FullyConnected dimension is walked -- 0 its full extent (the exchange has been done), 1 its interior only
// (the exchange is still in flight: everything interior tiles read), 2 its halo rows only (after the exchange)
template <class FT>
static void launch_shell(const GridD<FT>& g, const HaloBatch<FT>& hb, int comm_rows = 0) {
    ShellPlan P{};
    bool done[3] = {false, false, false};
    for (int D = 2; D >= 0; --D) {
        if (g.topo[D] != OB_PERIODIC) continue;
        ShellGroup& G = P.g[P.ng++];
        G.D = D;
        G.HD = -1;
        G.count = 1;
        for (int d = 0; d < 3; ++d) {
            if (d == D) { G.lo[d] = 0; G.n[d] = 2 * g.H[d]; }
            else if (g.topo[d] == OB_COMM && comm_rows == 1) { G.lo[d] = 1; G.n[d] = g.N[d]; }
            else if (g.topo[d] == OB_COMM && comm_rows == 2) { G.HD = d; G.lo[d] = 0; G.n[d] = 2 * g.H[d]; }
            else if (g.topo[d] == OB_FLAT || (g.topo[d] == OB_PERIODIC && done[d])) { G.lo[d] = 1; G.n[d] = g.N[d]; }
            else { G.lo[d] = 1 - g.H[d]; G.n[d] = g.N[d] + 2 * g.H[d]; }
            G.count *= G.n[d];
        }
        done[D] = true;
        P.total += G.count;
    }
    if (P.total == 0) return;
    fill_halo_shell_kernel<FT><<<cdiv(P.total, 256), 256, 0, stream()>>>(g, hb, P);
    OB_LAUNCH_CHECK();
}

// ---- halo exchange for a FullyConnected (slab-decomposed) dimension ---------------------------
// Reference: Distributed/halo_communication.jl:62-183 sends strided views per field and side with
// MPI.Isend/Irecv.  Here all fields' H boundary planes are packed into one contiguous buffer per
// side, exchanged with one grouped ncclSend/ncclRecv pair per side, and unpacked; the planes span
// the FULL extent of the other two dimensions so that edges and corners come out as in the
// single-process x -> y -> z sequence (fill_halo_regions_periodic.jl:15-31).
template <class FT, bool PACK>
__global__ void halo_pack_kernel(GridD<FT> g, HaloBatch<FT> hb, int d, int a, int b, int alo, int nA, int blo, int nB,
                                 FT* buf_lo, FT* buf_hi) {
    int ia = blockIdx.x * blockDim.x + threadIdx.x;
    int ib = blockIdx.y * blockDim.y + threadIdx.y;
    if (ia >= nA || ib >= nB) return;
    long long base = (alo + ia) * g.st[a] + (blo + ib) * g.st[b];
    long long s = g.st[d];
    int N = g.N[d], H = g.H[d];
    for (int n = 0; n < hb.n; ++n) {
        FT* f = hb.p0[n] + base;
        for (int h = 0; h < H; ++h) {
            long long q = (((long long)n * H + h) * nB + ib) * nA + ia;
            if (PACK) {
                buf_lo[q] = f[(1 + h) * s];               // rows 1..H       -> low-side neighbour's high halo
                buf_hi[q] = f[(N - H + 1 + h) * s];       // rows N-H+1..N   -> high-side neighbour's low halo
            } else {
                f[(1 - H + h) * s] = buf_lo[q];           // low halo  <- low-side neighbour's rows N-H+1..N
                f[(N + 1 + h) * s] = buf_hi[q];           // high halo <- high-side neighbour's rows 1..H
            }
        }
    }
}

namespace comm {
bool active(); int rank(); int size(); bool peer_access_ok();
void group_start(); void group_end();
void send(const void*, size_t, int); void recv(void*, size_t, int);
}

template <class FT>
static void exchange_halos(const GridD<FT>& g, const HaloBatch<FT>& hb, int d) {
    if (!comm::active()) throw Error("FullyConnected topology without an initialised communicator");
    int a = d == 0 ? 1 : 0, b = d == 2 ? 1 : 2;
    int ab[2] = {a, b}, lo[2], n[2];
    for (int q = 0; q < 2; ++q) {
        int e = ab[q];
        if (g.topo[e] == OB_FLAT) { lo[q] = 1; n[q] = 1; }
        else { lo[q] = 1 - g.H[e]; n[q] = g.N[e] + 2 * g.H[e] + 1; }
    }
    size_t elems = (size_t)hb.n * g.H[d] * n[0] * n[1], bytes = elems * sizeof(FT);
    static FT* buf[4] = {nullptr, nullptr, nullptr, nullptr};
    static size_t cap = 0;
    if (bytes > cap) {
        for (int q = 0; q < 4; ++q) { if (buf[q]) cudaFree(buf[q]); OB_CUDA(cudaMalloc(&buf[q], bytes)); }
        cap = bytes;
    }
    dim3 blk(a == 0 ? 64 : 16, a == 0 ? 4 : 16), grd(cdiv(n[0], blk.x), cdiv(n[1], blk.y));
    halo_pack_kernel<FT, true><<<grd, blk, 0, stream()>>>(g, hb, d, a, b, lo[0], n[0], lo[1], n[1], buf[0], buf[1]);
    OB_LAUNCH_CHECK();
    int R = comm::size(), r = comm::rank();
    int below = (r - 1 + R) % R, above = (r + 1) % R;
    comm::group_start();
    comm::send(buf[0], bytes, below);       // my low rows   -> neighbour below (its high halo)
    comm::send(buf[1], bytes, above);       // my high rows  -> neighbour above (its low halo)
    comm::recv(buf[3], bytes, above);       // high halo     <- neighbour above's low rows  (its first send)
    comm::recv(buf[2], bytes, below);       // low halo      <- neighbour below's high rows (its second send)
    comm::group_end();
    halo_pack_kernel<FT, false><<<grd, blk, 0, stream()>>>(g, hb, d, a, b, lo[0], n[0], lo[1], n[1], buf[2], buf[3]);
    OB_LAUNCH_CHECK();
}

// ---- the same exchange through peer memory (comm.cu: PeerLink) ------------------------------------------------
// The pack kernel stores the boundary planes straight into the neighbour's receive buffer over NVLink; flag words
// published / awaited by one-thread kernels order it with the neighbour's unpack.  `np` planes per side (np <= H);
// need_lo / need_hi: which of MY halos must be filled (every rank passes the same values, so need_hi means that
// every rank sends its bottom planes down).  The planes span the INTERIOR of the other dimensions: their halos are
// either not needed (wrap-around readers) or written afterwards by the shell fill.
namespace comm {
void peer_halo_prepare(size_t); void peer_halo_begin(); void peer_halo_check_pattern(bool, bool);
void* peer_halo_send_ptr(int); void* peer_halo_recv_ptr(int);
void peer_halo_signal(bool, bool); void peer_halo_wait(bool, bool);
}
template <class FT, bool PACK>
__global__ void halo_planes_kernel(GridD<FT> g, HaloBatch<FT> hb, int d, int a, int b, int nA, int nB, int np,
                                   FT* buf_lo, FT* buf_hi) {
    int ia = blockIdx.x * blockDim.x + threadIdx.x;
    int ib = blockIdx.y * blockDim.y + threadIdx.y;
    if (ia >= nA || ib >= nB) return;
    long long base = (1 + ia) * g.st[a] + (1 + ib) * g.st[b];
    long long s = g.st[d];
    int N = g.N[d];
    for (int n = 0; n < hb.n; ++n) {
        FT* f = hb.p0[n] + base;
        for (int h = 0; h < np; ++h) {
            long long q = (((long long)n * np + h) * nB + ib) * nA + ia;
            if (PACK) {
                if (buf_hi) buf_hi[q] = f[(1 + h) * s];              // my planes 1..np      -> the rank below's high halo
                if (buf_lo) buf_lo[q] = f[(N - np + 1 + h) * s];     // my planes N-np+1..N  -> the rank above's low halo
            } else {
                if (buf_lo) f[(1 - np + h) * s] = buf_lo[q];         // low halo  <- planes N-np+1..N of the rank below
                if (buf_hi) f[(N + 1 + h) * s] = buf_hi[q];          // high halo <- planes 1..np of the rank above
            }
        }
    }
}
static bool peer_halo_enabled() {
    static const bool off = getenv("OB200_NO_PEER_HALO") != nullptr;
    return !off && comm::active() && comm::peer_access_ok();
}
template <class FT>
void launch_exchange_planes(const GridD<FT>& g, const HaloBatch<FT>& hb, int d, int np, bool need_lo, bool need_hi) {
    if (hb.n == 0 || (!need_lo && !need_hi)) return;
    int a = d == 0 ? 1 : 0, b = d == 2 ? 1 : 2;
    int nA = g.N[a], nB = g.N[b];
    size_t bytes = (size_t)hb.n * np * nA * nB * sizeof(FT);
    // capacity for the largest exchange of this grid (MAXF fields, H planes) so that the link is set up once
    comm::peer_halo_prepare(std::max(bytes, (size_t)MAXF * g.H[d] * nA * nB * sizeof(FT)));
    comm::peer_halo_check_pattern(need_lo, need_hi);
    comm::peer_halo_begin();
    dim3 blk(a == 0 ? 64 : 16, a == 0 ? 4 : 16), grd(cdiv(nA, blk.x), cdiv(nB, blk.y));
    halo_planes_kernel<FT, true><<<grd, blk, 0, stream()>>>(g, hb, d, a, b, nA, nB, np,
        need_lo ? (FT*)comm::peer_halo_send_ptr(0) : nullptr, need_hi ? (FT*)comm::peer_halo_send_ptr(1) : nullptr);
    OB_LAUNCH_CHECK();
    comm::peer_halo_signal(need_lo, need_hi);
    comm::peer_halo_wait(need_lo, need_hi);
    halo_planes_kernel<FT, false><<<grd, blk, 0, stream()>>>(g, hb, d, a, b, nA, nB, np,
        need_lo ? (FT*)comm::peer_halo_recv_ptr(0) : nullptr, need_hi ? (FT*)comm::peer_halo_recv_ptr(1) : nullptr);
    OB_LAUNCH_CHECK();
}
template void launch_exchange_planes<float>(const GridD<float>&, const HaloBatch<float>&, int, int, bool, bool);
template void launch_exchange_planes<double>(const GridD<double>&, const HaloBatch<double>&, int, int, bool, bool);
template <class FT>
int single_comm_dim(const GridD<FT>& g) {       // the slab-decomposed dimension if there is exactly one, else -1
    int dc = -1;
    for (int d = 0; d < 3; ++d) if (g.topo[d] == OB_COMM) { if (dc >= 0) return -1; dc = d; }
    return dc;
}
template int single_comm_dim<float>(const GridD<float>&);
template int single_comm_dim<double>(const GridD<double>&);

// The same fill in two phases, for the overlap of the neighbour exchange with the interior tiles of the next tendency
// launch (halo_communication.jl:62-183 fills asynchronously; here the caller puts phase 1 on a side stream):
//   phase 0: the Periodic halos of the rows this rank owns -- all that tiles away from the slab boundary read;
//   phase 1: the exchange of the boundary planes through peer memory, then the Periodic halos of the received rows.
template <class FT>
bool halo_overlap_supported(const GridD<FT>& g) {
    const int dc = single_comm_dim(g);
    return dc >= 0 && peer_halo_enabled() && shell_fill_supported(g, true) && g.N[dc] >= g.H[dc];
}
template bool halo_overlap_supported<float>(const GridD<float>&);
template bool halo_overlap_supported<double>(const GridD<double>&);
template <class FT>
void launch_fill_halos_phase(const GridD<FT>& g, const HaloBatch<FT>& hb, int phase) {
    if (hb.n == 0) return;
    const int dc = single_comm_dim(g);
    if (phase == 0) { launch_shell<FT>(g, hb, 1); return; }
    launch_exchange_planes<FT>(g, hb, dc, g.H[dc], true, true);
    launch_shell<FT>(g, hb, 2);
}
template void launch_fill_halos_phase<float>(const GridD<float>&, const HaloBatch<float>&, int);
template void launch_fill_halos_phase<double>(const GridD<double>&, const HaloBatch<double>&, int);

template <class FT>
void launch_fill_halos(const GridD<FT>& g, const HaloBatch<FT>& hb) {
    if (hb.n == 0) return;
    if (shell_fill_supported(g, false)) { launch_shell<FT>(g, hb); return; }
    const int dc = single_comm_dim(g);
    if (dc >= 0 && peer_halo_enabled() && shell_fill_supported(g, true) && g.N[dc] >= g.H[dc]) {
        launch_exchange_planes<FT>(g, hb, dc, g.H[dc], true, true);
        launch_shell<FT>(g, hb);
        return;
    }
    // non-periodic first, then periodic / connected dimensions in x, y, z order (fill_halo_regions.jl:56-102)
    for (int pass = 0; pass < 2; ++pass)
        for (int d = 0; d < 3; ++d) {
            if (g.topo[d] == OB_FLAT) continue;
            bool per = g.topo[d] == OB_PERIODIC || g.topo[d] == OB_COMM;
            if ((pass == 0) == per) continue;
            if (per && g.H[d] == 0) continue;
            if (g.topo[d] == OB_COMM) { exchange_halos<FT>(g, hb, d); continue; }
            int a = d == 0 ? 1 : 0, b = d == 2 ? 1 : 2;
            int lo[2], hi[2], ab[2] = {a, b};
            for (int q = 0; q < 2; ++q) {
                int e = ab[q];
                if (g.topo[e] == OB_FLAT) { lo[q] = hi[q] = 1; }
                else if (per) { lo[q] = 1 - g.H[e]; hi[q] = g.N[e] + g.H[e] + 1; }
                else { lo[q] = 1; hi[q] = g.N[e]; }
            }
            dim3 blk(a == 0 ? 64 : 16, a == 0 ? 4 : 16);
            dim3 grd(cdiv(hi[0] - lo[0] + 1, blk.x), cdiv(hi[1] - lo[1] + 1, blk.y));
            static_assert(sizeof(GridD<double>) + sizeof(HaloBatch<double>) + 6 * sizeof(int) <= 4096,
                          "fill_halo_kernel parameters must stay within the 4 KB kernel-parameter space");
            fill_halo_kernel<FT><<<grd, blk, 0, stream()>>>(g, hb, d, a, b, lo[0], hi[0], lo[1], hi[1]);
            OB_LAUNCH_CHECK();
        }
}
template void launch_fill_halos<float>(const GridD<float>&, const HaloBatch<float>&);
template void launch_fill_halos<double>(const GridD<double>&, const HaloBatch<double>&);

// =============================================================================================
// general tendency kernel, one thread per cell, fused substep (out of place)
// =============================================================================================
template <class FT>
struct TendArgs {
    const FT* U[3];
    const FT* psi;
    const FT* pHY;
    Buoy<FT> b;
    FT* Gn;
    const FT* Gm;
    FT* psi_new;
    Substep<FT> ss;
    FluxBC<FT> fbc;
    int comp;
    int closure_only;      // G^n = -div(tau) / -div(q) of the closure alone (the fused kernel adds the rest, tendency_fused.cu)
    int bg_acc;            // background-only mode (tendency_shared_kernel BG = 2): add to G^n instead of overwriting it
};

// COMP (0, 1, 2 = u, v, w; 3 = any tracer) is a template parameter so that the staggering flags of every operator in
// the inlined call tree (locations, which spacings and areas, which directions interpolate) are compile-time constants
template <class FT, int COMP, bool BG = false>
__global__ void __launch_bounds__(128) tendency_general_kernel(const __grid_constant__ Phys<FT> P, const __grid_constant__ TendArgs<FT> A) {
    const GridD<FT>& g = P.g;
    int i = 1 + blockIdx.x * blockDim.x + threadIdx.x;
    int j = 1 + blockIdx.y * blockDim.y + threadIdx.y;
    int k = 1 + blockIdx.z;
    if (i > g.N[0] || j > g.N[1]) return;
    Pt q;
    q.i[0] = i; q.i[1] = j; q.i[2] = k;
    q.p = i * g.st[0] + j * g.st[1] + k * g.st[2];
    const FT* U[3] = {A.U[0], A.U[1], A.U[2]};
    FT G = tendency<FT, BG>(P, COMP == 3 ? A.comp : COMP, U, A.psi, A.pHY, A.b, q);
    // apply_x/y/z_bcs! (apply_flux_bcs.jl:35-160): constant Flux BCs of this field
    int l[3] = {OB_C, OB_C, OB_C};
    if (COMP < 3) l[COMP] = OB_F;
#pragma unroll
    for (int d = 0; d < 3; ++d) {
        if (g.topo[d] != OB_BOUNDED) continue;
        int lf[3] = {l[0], l[1], l[2]};
        lf[d] = l[d] == OB_C ? OB_F : OB_C;
        if (A.fbc.kind[2 * d] == 2 && q.i[d] == 1 && A.fbc.val[2 * d] != FT(0))
            G += A.fbc.val[2 * d] * areaA(g, d, q, lf[0], lf[1], lf[2]) / volume(g, q, l[0], l[1], l[2]);
        if (A.fbc.kind[2 * d + 1] == 2 && q.i[d] == g.N[d] && A.fbc.val[2 * d + 1] != FT(0))
            G -= A.fbc.val[2 * d + 1] * areaA(g, d, sh(g, q, d, 1), lf[0], lf[1], lf[2]) /
                 volume(g, q, l[0], l[1], l[2]);
    }
    A.Gn[q.p] = G;
    const Substep<FT>& s = A.ss;
    if (s.mode == SUB_RK3_FIRST) A.psi_new[q.p] = A.psi[q.p] + s.c1 * G;
    else if (s.mode == SUB_RK3) A.psi_new[q.p] = A.psi[q.p] + s.dt * (s.c1 * G + s.c2 * A.Gm[q.p]);
    else if (s.mode == SUB_AB2) A.psi_new[q.p] = A.psi[q.p] + s.dt * (s.c1 * G - s.c2 * A.Gm[q.p]);
}

// =============================================================================================
// array Flux boundary conditions: one boundary-plane pass per Bounded dimension after the tendency kernels of every path
// (apply_x/y/z_bcs!, apply_flux_bcs.jl:35-160, run in the reference as a separate step after the interior tendencies, in
// dimension order).  One thread per tangential point (ia, ib) walks the fields and both sides of dimension d in sequence, so a
// cell that is first and last at once (N = 1) gets both contributions in the reference's order.  The sum and the substep are
// the expressions of tendency_general_kernel above.
// =============================================================================================
template <class FT, int d>
__global__ void __launch_bounds__(128) boundary_flux_kernel(const GridD<FT> g, const BoundaryFluxes<FT> A, int na, int nb) {
    constexpr int a = d == 0 ? 1 : 0, b = d == 2 ? 1 : 2;      // tangential dimensions (compile-time: no local-memory indexing)
    const int ia = 1 + blockIdx.x * blockDim.x + threadIdx.x;
    const int ib = 1 + blockIdx.y * blockDim.y + threadIdx.y;
    if (ia > na || ib > nb) return;
    const long long t = (ia - 1) + (long long)(ib - 1) * na;       // Q[ia, ib], column-major
    Pt q;
    q.i[a] = ia; q.i[b] = ib;
    const Substep<FT>& s = A.ss;
    for (int n = 0; n < A.n; ++n) {
        const int c = A.comp[n];
        const int l[3] = {c == 0 ? OB_F : OB_C, c == 1 ? OB_F : OB_C, c == 2 ? OB_F : OB_C};
        int lf[3] = {l[0], l[1], l[2]};
        lf[d] = l[d] == OB_C ? OB_F : OB_C;
        for (int side = 0; side < 2; ++side) {
            const FT* Q = A.Q[n][side];
            if (!Q) continue;
            q.i[d] = side == 0 ? 1 : g.N[d];
            q.p = q.i[0] * g.st[0] + q.i[1] * g.st[1] + q.i[2] * g.st[2];
            FT G = A.Gn[n][q.p];
            if (side == 0) G += Q[t] * areaA(g, d, q, lf[0], lf[1], lf[2]) / volume(g, q, l[0], l[1], l[2]);
            else G -= Q[t] * areaA(g, d, sh(g, q, d, 1), lf[0], lf[1], lf[2]) / volume(g, q, l[0], l[1], l[2]);
            A.Gn[n][q.p] = G;
            const FT* psi = A.psi[n];
            FT* psi_new = A.psi_new[n];
            if (s.mode == SUB_RK3_FIRST) psi_new[q.p] = psi[q.p] + s.c1 * G;
            else if (s.mode == SUB_RK3) psi_new[q.p] = psi[q.p] + s.dt * (s.c1 * G + s.c2 * A.Gm[n][q.p]);
            else if (s.mode == SUB_AB2) psi_new[q.p] = psi[q.p] + s.dt * (s.c1 * G - s.c2 * A.Gm[n][q.p]);
        }
    }
}

template <class FT>
void launch_boundary_fluxes(const GridD<FT>& g, int d, const BoundaryFluxes<FT>& A) {
    if (A.n == 0) return;
    const int a = d == 0 ? 1 : 0, b = d == 2 ? 1 : 2;
    const int na = g.topo[a] == OB_FLAT ? 1 : g.N[a], nb = g.topo[b] == OB_FLAT ? 1 : g.N[b];
    dim3 blk(a == 0 ? 32 : 16, a == 0 ? 4 : 8);
    dim3 grd(cdiv(na, blk.x), cdiv(nb, blk.y));
    if (d == 0) boundary_flux_kernel<FT, 0><<<grd, blk, 0, stream()>>>(g, A, na, nb);
    else if (d == 1) boundary_flux_kernel<FT, 1><<<grd, blk, 0, stream()>>>(g, A, na, nb);
    else boundary_flux_kernel<FT, 2><<<grd, blk, 0, stream()>>>(g, A, na, nb);
    OB_LAUNCH_CHECK();
}
template void launch_boundary_fluxes<float>(const GridD<float>&, int, const BoundaryFluxes<float>&);
template void launch_boundary_fluxes<double>(const GridD<double>&, int, const BoundaryFluxes<double>&);

// =============================================================================================
// general tendency kernel with SHARED faces (any scheme / closure / BCs on a 3-D grid)
// The kernel above evaluates both faces of every cell in every direction (as the reference does,
// momentum_advection_operators.jl:52-56): each face flux is computed twice.  Here a block of 32 x 8 threads walks
// up in k and every thread evaluates ONE face per direction -- advective + viscous / diffusive flux summed -- of
// its own position; the other face of a cell comes from the neighbouring thread: along x by a warp shuffle, along y
// through shared memory, along z from the previous level kept in a register.  Tiles overlap by one column and one
// row (31 x 7 cells are finished per block), which replaces every special case at tile edges.  Same operator
// functions (physics.cuh) as the kernel above; the divergence of the summed fluxes differs from the sum of the two
// divergences by rounding only.
// =============================================================================================
// SPEC = 1: the configuration class of BASELINE config 3 (x, y Periodic and regular, z Bounded, WENO5, vertical gravity,
// explicit closure): the kernel works on a LOCAL copy of the physics descriptor whose flags are overwritten with these
// constants, so that after inlining every run-time scheme / topology / regularity branch of the operator tree folds away.
// CO = 1: closure-only (TendArgs::closure_only) as a compile-time flag, so that the advection operators are not part of the
// kernel at all, with 4 resident blocks per SM (64 registers; C3 with AMD: 3 blocks 64.3, 4 blocks 60.5, 5 blocks 62.0 ms per step)
// BG = 1: every face flux also carries the background fluxes F(U_bg, ψ) + F(U, ψ_bg) (Phys::bg, bgU).  BG = 2: background-only,
// G^n = (or +=, TendArgs::bg_acc) -div of those fluxes alone, the analogue of CO for the fused kernel's accumulate form
template <class FT, int COMP, int SPEC, int CO = 0, int BG = 0>
__global__ void __launch_bounds__(256, (CO || BG == 2 ? 4 : 3)) tendency_shared_kernel(const __grid_constant__ Phys<FT> Pin, const __grid_constant__ TendArgs<FT> A, int Kc) {
    Phys<FT> Pl;
    if constexpr (SPEC == 1) {
        Pl = Pin;
        Pl.g.topo[0] = OB_PERIODIC; Pl.g.topo[1] = OB_PERIODIC; Pl.g.topo[2] = OB_BOUNDED;
        Pl.g.regular[0] = 1; Pl.g.regular[1] = 1;
        Pl.scheme = ADV_WENO5; Pl.buffer = 2;
        Pl.wc[0][0] = nullptr; Pl.wc[0][1] = nullptr; Pl.wc[1][0] = nullptr; Pl.wc[1][1] = nullptr;
        Pl.tilted = 0; Pl.vitd = 0;
    }
    const Phys<FT>& P = SPEC ? Pl : Pin;
    const GridD<FT>& g = P.g;
    constexpr int TXS = 32, TYS = 8;
    constexpr int B = COMP < 3 ? COMP : 3;
    // pairing along direction d: LOW = the cell needs f(q) - f(q-1) (its own face and the previous thread's),
    // HIGH = f(q+1) - f(q).  Momentum: LOW along its own direction, HIGH otherwise; tracers: HIGH everywhere.
    constexpr bool XLOW = B == 0, YLOW = B == 1, ZLOW = B == 2;
    __shared__ FT sF[2][TYS][TXS];
    const int tx = threadIdx.x, ty = threadIdx.y;
    const int i = (XLOW ? 0 : 1) + blockIdx.x * (TXS - 1) + tx;
    const int j = (YLOW ? 0 : 1) + blockIdx.y * (TYS - 1) + ty;
    const int k0 = 1 + blockIdx.z * Kc, k1 = min(g.N[2], k0 + Kc - 1);
    const bool outx = (XLOW ? tx >= 1 : tx <= TXS - 2) && i >= 1 && i <= g.N[0];
    const bool outy = (YLOW ? ty >= 1 : ty <= TYS - 2) && j >= 1 && j <= g.N[1];
    const bool cell = outx && outy;
    const bool need_x = outy && i <= g.N[0] + 1, need_y = outx && j <= g.N[1] + 1;
    const FT* U[3] = {A.U[0], A.U[1], A.U[2]};
    const int comp = COMP == 3 ? A.comp : COMP;
    const bool visc = BG != 2 && P.closure != CLO_NONE, adv = !CO && BG != 2 && P.scheme != ADV_NONE && !A.closure_only;
    const FT* const* Ub = Pin.bgU;
    const FT* psib = BG ? Pin.bg[comp] : nullptr;
    const FT kappa = COMP == 3 ? Pin.kappa[comp - 3] : FT(0);
    const FT* kappae = COMP == 3 ? Pin.kappae[comp - 3] : nullptr;
    auto face = [&](int d, Pt q) -> FT {       // area-weighted advective + viscous / diffusive flux at q along d
        FT f = FT(0);
        if (COMP < 3) {
            if (adv) f = momentum_flux(P, d, B, U[d], A.psi, q);
            if (visc) f = f + viscous_Aflux(P, B, d, U, q);
        } else {
            if (adv) f = tracer_flux(P, d, U[d], A.psi, q);
            if (visc) f = f + diffusive_Aflux(P, d, kappa, A.psi, q, kappae);
        }
        return f;
    };
    // the same with the background fluxes F(U_bg, ψ) + F(U, ψ_bg) (BG != 0).  A separate lambda, so that the BG = 0 kernels keep
    // their code; always inlined, since out of line the call would keep the physics descriptor on the stack
    auto face_bg = [&](int d, Pt q) __attribute__((always_inline)) -> FT {
        FT f = FT(0);
        if (COMP < 3) {
            if (adv) f = momentum_flux(P, d, B, U[d], A.psi, q);
            if (Ub[0]) f = f + momentum_flux(P, d, B, Ub[d], A.psi, q);
            if (psib) f = f + momentum_flux(P, d, B, U[d], psib, q);
            if (visc) f = f + viscous_Aflux(P, B, d, U, q);
        } else {
            if (adv) f = tracer_flux(P, d, U[d], A.psi, q);
            if (Ub[0]) f = f + tracer_flux(P, d, Ub[d], A.psi, q);
            if (psib) f = f + tracer_flux(P, d, U[d], psib, q);
            if (visc) f = f + diffusive_Aflux(P, d, kappa, A.psi, q, kappae);
        }
        return f;
    };
    Pt q;
    q.i[0] = i; q.i[1] = j; q.i[2] = k0;
    q.p = i * g.st[0] + j * g.st[1] + k0 * g.st[2];
    FT Fz_carry = FT(0);
    if (cell) Fz_carry = BG ? face_bg(2, ZLOW ? sh(g, q, 2, -1) : q) : face(2, ZLOW ? sh(g, q, 2, -1) : q);
    for (int k = k0; k <= k1; ++k) {
        const int buf = (k - k0) & 1;
        FT Fx = FT(0), Fy = FT(0), dFz = FT(0);
        if (need_x) Fx = BG ? face_bg(0, q) : face(0, q);
        if (need_y) Fy = BG ? face_bg(1, q) : face(1, q);
        sF[buf][ty][tx] = Fy;
        if (cell) {
            FT Fz_new = BG ? face_bg(2, ZLOW ? q : sh(g, q, 2, 1)) : face(2, ZLOW ? q : sh(g, q, 2, 1));
            dFz = Fz_new - Fz_carry;
            Fz_carry = Fz_new;
        }
        const FT Fxn = XLOW ? __shfl_up_sync(0xffffffffu, Fx, 1) : __shfl_down_sync(0xffffffffu, Fx, 1);
        __syncthreads();
        if (cell) {
            const FT dFx = XLOW ? (Fx - Fxn) : (Fxn - Fx);
            const FT Fyn = sF[buf][YLOW ? ty - 1 : ty + 1][tx];
            const FT dFy = YLOW ? (Fy - Fyn) : (Fyn - Fy);
            int l[3] = {OB_C, OB_C, OB_C};
            if (COMP < 3) l[COMP] = OB_F;
            FT G = -((1 / volume(g, q, l[0], l[1], l[2])) * ((dFx + dFy) + dFz));
            if (BG == 2) {
                A.Gn[q.p] = A.bg_acc ? A.Gn[q.p] + G : G;
            } else if (CO || A.closure_only) {
                A.Gn[q.p] = G;
            } else {
            if (COMP == 0) {
                if (P.fplane) {          // x_f_cross_U = -f ℑxyᶠᶜᵃ(v)   (f_plane.jl:42)
                    FT a0 = IF(g, U[1], q, 0);
                    FT v = g.topo[1] == OB_FLAT ? a0 : FT(0.5) * (a0 + IF(g, U[1], sh(g, q, 1, 1), 0));
                    G = G - (-P.f * v);
                }
                if (A.pHY) G = G - deriv(g, A.pHY, q, 0, OB_F);
            } else if (COMP == 1) {
                if (P.fplane) {          // y_f_cross_U = f ℑxyᶜᶠᵃ(u)    (f_plane.jl:43)
                    FT a1 = IC(g, U[0], q, 0);
                    FT u = g.topo[1] == OB_FLAT ? a1 : FT(0.5) * (IC(g, U[0], sh(g, q, 1, -1), 0) + a1);
                    G = G - (P.f * u);
                }
                if (A.pHY) G = G - deriv(g, A.pHY, q, 1, OB_F);
            }
            if (COMP < 2 && P.tilted && A.b.mode) G = G + P.ghat[COMP] * buoyancy_at(A.b, q.p);      // x/y_dot_g_b (g_dot_b.jl:1-3)
            // + forcing, last in the sum (the descriptor read from the kernel parameter: `comp` may be run-time data)
            if (Pin.frc[comp].on) G = G + relaxation(Pin.frc[comp], q.i[0], q.i[1], q.i[2], A.psi[q.p]);
            // apply_x/y/z_bcs! (apply_flux_bcs.jl:35-160): constant Flux BCs of this field
#pragma unroll
            for (int d = 0; d < 3; ++d) {
                if (g.topo[d] != OB_BOUNDED) continue;
                int lf[3] = {l[0], l[1], l[2]};
                lf[d] = l[d] == OB_C ? OB_F : OB_C;
                if (A.fbc.kind[2 * d] == 2 && q.i[d] == 1 && A.fbc.val[2 * d] != FT(0))
                    G += A.fbc.val[2 * d] * areaA(g, d, q, lf[0], lf[1], lf[2]) / volume(g, q, l[0], l[1], l[2]);
                if (A.fbc.kind[2 * d + 1] == 2 && q.i[d] == g.N[d] && A.fbc.val[2 * d + 1] != FT(0))
                    G -= A.fbc.val[2 * d + 1] * areaA(g, d, sh(g, q, d, 1), lf[0], lf[1], lf[2]) /
                         volume(g, q, l[0], l[1], l[2]);
            }
            A.Gn[q.p] = G;
            const Substep<FT>& ss = A.ss;
            if (ss.mode == SUB_RK3_FIRST) A.psi_new[q.p] = A.psi[q.p] + ss.c1 * G;
            else if (ss.mode == SUB_RK3) A.psi_new[q.p] = A.psi[q.p] + ss.dt * (ss.c1 * G + ss.c2 * A.Gm[q.p]);
            else if (ss.mode == SUB_AB2) A.psi_new[q.p] = A.psi[q.p] + ss.dt * (ss.c1 * G - ss.c2 * A.Gm[q.p]);
            }
        }
        q = sh(g, q, 2, 1);
    }
}

template <class FT>
bool closure_only_supported(const Phys<FT>& P) {
    if (P.closure == CLO_NONE) return false;
    for (int d = 0; d < 3; ++d) if (P.g.topo[d] == OB_FLAT || P.g.N[d] < 2) return false;
    return true;
}
template bool closure_only_supported<float>(const Phys<float>&);
template bool closure_only_supported<double>(const Phys<double>&);
template <class FT>
bool background_only_supported(const Phys<FT>& P) {
    if (P.scheme == ADV_NONE) return false;
    for (int d = 0; d < 3; ++d) if (P.g.topo[d] == OB_FLAT || P.g.N[d] < 2) return false;
    return true;
}
template bool background_only_supported<float>(const Phys<float>&);
template bool background_only_supported<double>(const Phys<double>&);

template <class FT>
void launch_tendency_general(const Phys<FT>& P, int comp, const FT* const U[3], const FT* psi,
                             const FT* pHY, const Buoy<FT>& b, const FluxBC<FT>& fbc, FT* Gn,
                             const FT* Gm, FT* psi_new, const Substep<FT>& ss, bool closure_only, int background_only) {
    TendArgs<FT> A;
    for (int d = 0; d < 3; ++d) A.U[d] = U[d];
    A.psi = psi; A.pHY = pHY; A.b = b; A.Gn = Gn; A.Gm = Gm; A.psi_new = psi_new;
    A.ss = ss; A.fbc = fbc; A.comp = comp; A.closure_only = closure_only ? 1 : 0; A.bg_acc = background_only == 2 ? 1 : 0;
    const bool bg = has_background(P, comp);
    // shared-face variant: 3-D grids (every direction has two faces to pair) with a halo wide enough for the one
    // extra face position per direction
    bool shared = P.scheme != ADV_NONE || P.closure != CLO_NONE;
    for (int d = 0; d < 3; ++d) shared = shared && P.g.topo[d] != OB_FLAT && P.g.N[d] >= 2;
    if (closure_only && !shared) throw Error("closure-only tendencies need the shared-face kernel (3-D grid)");
    if (background_only && !(shared && background_only_supported(P)))
        throw Error("background-only tendencies need the shared-face kernel (3-D grid, an advection scheme)");
    const bool spec = P.g.topo[0] == OB_PERIODIC && P.g.topo[1] == OB_PERIODIC && P.g.topo[2] == OB_BOUNDED &&
                      P.g.regular[0] && P.g.regular[1] && P.scheme == ADV_WENO5 && P.buffer == 2 && !P.tilted && !P.vitd &&
                      !P.wc[0][0] && !P.wc[0][1] && !P.wc[1][0] && !P.wc[1][1];
    if (shared) {
        const int Kc = 32;
        dim3 bs(32, 8, 1), gs(cdiv(P.g.N[0], 31), cdiv(P.g.N[1], 7), cdiv(P.g.N[2], Kc));
        switch (comp) {
#define SHK(C, S) do { if (closure_only) tendency_shared_kernel<FT, C, S, 1><<<gs, bs, 0, stream()>>>(P, A, Kc); \
                       else if (background_only) tendency_shared_kernel<FT, C, S, 0, 2><<<gs, bs, 0, stream()>>>(P, A, Kc); \
                       else if (bg) tendency_shared_kernel<FT, C, S, 0, 1><<<gs, bs, 0, stream()>>>(P, A, Kc); \
                       else tendency_shared_kernel<FT, C, S, 0><<<gs, bs, 0, stream()>>>(P, A, Kc); } while (0)
            case 0: if (spec) SHK(0, 1); else SHK(0, 0); break;
            case 1: if (spec) SHK(1, 1); else SHK(1, 0); break;
            case 2: if (spec) SHK(2, 1); else SHK(2, 0); break;
            default: if (spec) SHK(3, 1); else SHK(3, 0); break;
#undef SHK
        }
        OB_LAUNCH_CHECK();
        return;
    }
    dim3 blk(32, 4, 1);
    dim3 grd(cdiv(P.g.N[0], 32), cdiv(P.g.N[1], 4), P.g.N[2]);
#define GK(C) do { if (bg) tendency_general_kernel<FT, C, true><<<grd, blk, 0, stream()>>>(P, A); \
                   else tendency_general_kernel<FT, C><<<grd, blk, 0, stream()>>>(P, A); } while (0)
    switch (comp) {
        case 0: GK(0); break;
        case 1: GK(1); break;
        case 2: GK(2); break;
        default: GK(3); break;
    }
#undef GK
    OB_LAUNCH_CHECK();
}
template void launch_tendency_general<float>(const Phys<float>&, int, const float* const[3], const float*,
                                             const float*, const Buoy<float>&, const FluxBC<float>&, float*,
                                             const float*, float*, const Substep<float>&, bool, int);
template void launch_tendency_general<double>(const Phys<double>&, int, const double* const[3], const double*,
                                              const double*, const Buoy<double>&, const FluxBC<double>&, double*,
                                              const double*, double*, const Substep<double>&, bool, int);

// =============================================================================================
// pressure source term: rhs = div(U*) / dt (x Δzᶜ for the tridiagonal solver)
// solve_for_pressure.jl:15-33, divergence_operators.jl:16-19
// =============================================================================================
template <class FT>
__device__ __forceinline__ FT div_ccc(const GridD<FT>& g, const FT* u, const FT* v, const FT* w, Pt q) {
    FT t[3];
    const FT* U[3] = {u, v, w};
#pragma unroll
    for (int d = 0; d < 3; ++d) {
        if (g.topo[d] == OB_FLAT) { t[d] = FT(0); continue; }
        int l[3] = {OB_C, OB_C, OB_C};
        l[d] = OB_F;
        Pt q1 = sh(g, q, d, 1);
        t[d] = areaA(g, d, q1, l[0], l[1], l[2]) * U[d][q1.p] - areaA(g, d, q, l[0], l[1], l[2]) * U[d][q.p];
    }
    return (1 / volume(g, q, OB_C, OB_C, OB_C)) * ((t[0] + t[1]) + t[2]);
}

template <class FT, class CT>
__global__ void pressure_rhs_kernel(GridD<FT> g, const FT* u, const FT* v, const FT* w, FT dt,
                                    bool times_dz, CT* rhs) {
    int i = 1 + blockIdx.x * blockDim.x + threadIdx.x;
    int j = 1 + blockIdx.y * blockDim.y + threadIdx.y;
    int k = 1 + blockIdx.z;
    if (i > g.N[0] || j > g.N[1]) return;
    Pt q;
    q.i[0] = i; q.i[1] = j; q.i[2] = k;
    q.p = i * g.st[0] + j * g.st[1] + k * g.st[2];
    FT dv = div_ccc(g, u, v, w, q);
    FT r = times_dz ? (spacing(g, 2, OB_C, k) * dv) / dt : dv / dt;
    CT c;
    c.x = r; c.y = 0;
    rhs[(i - 1) + (long long)g.N[0] * ((j - 1) + (long long)g.N[1] * (k - 1))] = c;
}
template <class FT, class CT>
void launch_pressure_rhs(const GridD<FT>& g, const FT* u, const FT* v, const FT* w, FT dt,
                         bool times_dz, CT* rhs) {
    dim3 blk(64, 4, 1), grd(cdiv(g.N[0], 64), cdiv(g.N[1], 4), g.N[2]);
    pressure_rhs_kernel<FT, CT><<<grd, blk, 0, stream()>>>(g, u, v, w, dt, times_dz, rhs);
    OB_LAUNCH_CHECK();
}
template void launch_pressure_rhs<float, float2>(const GridD<float>&, const float*, const float*, const float*,
                                                 float, bool, float2*);
template void launch_pressure_rhs<double, double2>(const GridD<double>&, const double*, const double*,
                                                   const double*, double, bool, double2*);

// _pressure_correct_velocities! pressure_correction.jl:34-40
template <class FT>
__global__ void pressure_correct_kernel(GridD<FT> g, FT* u, FT* v, FT* w, const FT* p, FT dt) {
    int i = 1 + blockIdx.x * blockDim.x + threadIdx.x;
    int j = 1 + blockIdx.y * blockDim.y + threadIdx.y;
    int k = 1 + blockIdx.z;
    if (i > g.N[0] || j > g.N[1]) return;
    Pt q;
    q.i[0] = i; q.i[1] = j; q.i[2] = k;
    q.p = i * g.st[0] + j * g.st[1] + k * g.st[2];
    u[q.p] -= deriv(g, p, q, 0, OB_F) * dt;
    v[q.p] -= deriv(g, p, q, 1, OB_F) * dt;
    w[q.p] -= deriv(g, p, q, 2, OB_F) * dt;
}
// The same on a grid whose non-Flat dimensions are all Periodic and regular: p is read with wrap-around, so its
// halos need not be valid (the fill_halo_regions! of pressure_correction.jl:17 is merged into the single
// shell fill at the end of the stage).
template <class FT>
__global__ void __launch_bounds__(256) pressure_correct_periodic_kernel(GridD<FT> g, FT* u, FT* v, FT* w, const FT* p, FT dt) {
    int i = 1 + blockIdx.x * blockDim.x + threadIdx.x;
    int j = 1 + blockIdx.y * blockDim.y + threadIdx.y;
    int k = 1 + blockIdx.z;
    if (i > g.N[0] || j > g.N[1]) return;
    const int id[3] = {i, j, k};
    const long long q = i * g.st[0] + j * g.st[1] + k * g.st[2];
    const FT pc = p[q];
    FT* const U[3] = {u, v, w};
#pragma unroll
    for (int d = 0; d < 3; ++d) {
        if (g.topo[d] == OB_FLAT) { U[d][q] -= (FT(0) / g.d[d]) * dt; continue; }
        // Periodic: wrap; slab-decomposed: the low halo plane (exchanged by the caller)
        const long long qm = q - g.st[d] + (id[d] == 1 && g.topo[d] == OB_PERIODIC ? (long long)g.N[d] * g.st[d] : 0);
        U[d][q] -= ((pc - p[qm]) / g.d[d]) * dt;
    }
}
// two cells per thread (aligned 16-byte / 8-byte vector accesses: interior rows start 32-byte aligned) and two levels
// per thread (the pressure of the lower level is reused from registers): fewer, wider memory instructions in flight
template <class FT> struct Vec2;
template <> struct Vec2<double> { using T = double2; };
template <> struct Vec2<float> { using T = float2; };
template <class FT>
__global__ void __launch_bounds__(128) pressure_correct_periodic_v2_kernel(GridD<FT> g, FT* u, FT* v, FT* w, const FT* p, FT dt) {
    using V2 = typename Vec2<FT>::T;
    const int i = 1 + 2 * (blockIdx.x * blockDim.x + threadIdx.x);
    const int j = 1 + blockIdx.y * blockDim.y + threadIdx.y;
    const int k0 = 1 + 2 * blockIdx.z;
    if (i > g.N[0] || j > g.N[1]) return;
    const long long sy = g.st[1], sz = g.st[2];
    const long long q0 = i + j * sy + k0 * sz;
    const long long wy = j == 1 && g.topo[1] == OB_PERIODIC ? (long long)g.N[1] * sy : 0;
    const long long wx = i == 1 && g.topo[0] == OB_PERIODIC ? (long long)g.N[0] : 0;
    const long long wz = k0 == 1 && g.topo[2] == OB_PERIODIC ? (long long)g.N[2] * sz : 0;
    // loads of both levels first
    V2 pc[2], py[2], uu[2], vv[2], ww[2];
    FT pxm[2];
    const V2 pzm = *reinterpret_cast<const V2*>(p + q0 - sz + wz);
#pragma unroll
    for (int e = 0; e < 2; ++e) {
        const long long q = q0 + e * sz;
        pc[e] = *reinterpret_cast<const V2*>(p + q);
        py[e] = *reinterpret_cast<const V2*>(p + q - sy + wy);
        pxm[e] = p[q - 1 + wx];
        uu[e] = *reinterpret_cast<const V2*>(u + q);
        vv[e] = *reinterpret_cast<const V2*>(v + q);
        ww[e] = *reinterpret_cast<const V2*>(w + q);
    }
#pragma unroll
    for (int e = 0; e < 2; ++e) {
        const long long q = q0 + e * sz;
        const V2 pz = e == 0 ? pzm : pc[0];
        uu[e].x -= ((pc[e].x - pxm[e]) / g.d[0]) * dt;  uu[e].y -= ((pc[e].y - pc[e].x) / g.d[0]) * dt;
        vv[e].x -= ((pc[e].x - py[e].x) / g.d[1]) * dt; vv[e].y -= ((pc[e].y - py[e].y) / g.d[1]) * dt;
        const FT dz = spacing(g, 2, OB_F, k0 + e);          // regular: g.d[2]; stretched: the level's own Δz at the face
        ww[e].x -= ((pc[e].x - pz.x) / dz) * dt;        ww[e].y -= ((pc[e].y - pz.y) / dz) * dt;
        *reinterpret_cast<V2*>(u + q) = uu[e];
        *reinterpret_cast<V2*>(v + q) = vv[e];
        *reinterpret_cast<V2*>(w + q) = ww[e];
    }
}
template <class FT>
bool periodic_wrap_supported(const GridD<FT>& g) {
    bool any = false;
    for (int d = 0; d < 3; ++d) {
        if (g.topo[d] == OB_FLAT) continue;
        if (g.topo[d] == OB_COMM) {       // one slab-decomposed dimension, exchanged through peer memory
            if (single_comm_dim(g) != d || !peer_halo_enabled() || !g.regular[d] || g.N[d] < 2 * g.H[d]) return false;
            continue;
        }
        if (g.topo[d] != OB_PERIODIC || !g.regular[d] || g.N[d] < 2 * g.H[d]) return false;
        any = true;
    }
    return any;
}
template bool periodic_wrap_supported<float>(const GridD<float>&);
template bool periodic_wrap_supported<double>(const GridD<double>&);

template <class FT>
void launch_pressure_correct(const GridD<FT>& g, FT* u, FT* v, FT* w, const FT* p, FT dt, bool periodic_wrap) {
    dim3 blk(64, 4, 1), grd(cdiv(g.N[0], 64), cdiv(g.N[1], 4), g.N[2]);
    // v2: two cells x two levels per thread.  With valid halos of p (not periodic_wrap) it serves every 3-D grid with regular
    // x, y and even Nx, Nz: Periodic dimensions are read with wrap-around (the same values), the others from their halos
    bool v2 = g.N[0] % 2 == 0 && g.N[2] % 2 == 0 && g.regular[0] && g.regular[1] && (periodic_wrap || g.regular[2] || g.dF[2]);
    for (int d = 0; d < 3; ++d) v2 = v2 && g.topo[d] != OB_FLAT;      // 3-D only: all three corrections active
    if (v2) {
        dim3 b2(32, 4, 1), g2(cdiv(g.N[0] / 2, 32), cdiv(g.N[1], 4), g.N[2] / 2);
        pressure_correct_periodic_v2_kernel<FT><<<g2, b2, 0, stream()>>>(g, u, v, w, p, dt);
    } else if (periodic_wrap) pressure_correct_periodic_kernel<FT><<<grd, blk, 0, stream()>>>(g, u, v, w, p, dt);
    else pressure_correct_kernel<FT><<<grd, blk, 0, stream()>>>(g, u, v, w, p, dt);
    OB_LAUNCH_CHECK();
}
template void launch_pressure_correct<float>(const GridD<float>&, float*, float*, float*, const float*, float, bool);
template void launch_pressure_correct<double>(const GridD<double>&, double*, double*, double*, const double*, double, bool);

// _update_hydrostatic_pressure! update_hydrostatic_pressure.jl:10-18 : one column per thread, top to bottom, same
// summation order as the reference.  The column is walked in batches of HU levels whose loads are issued
// together (the serial k recurrence otherwise exposes one DRAM latency per level: ncu r1d showed 20 % of peak
// DRAM throughput with long-scoreboard as the only stall).
// WRAP (z Periodic): b[Nz+1] is read as b[1], so the tracer's halos need not be valid.
template <class FT, bool WRAP, int BMODE>
__global__ void __launch_bounds__(64) hydrostatic_kernel(GridD<FT> g, const Buoy<FT> b, FT gz, bool tilted, FT* pHY) {
    constexpr int HU = 16;
    int i = 1 + blockIdx.x * blockDim.x + threadIdx.x;
    int j = 1 + blockIdx.y * blockDim.y + threadIdx.y;
    if (i > g.N[0] || j > g.N[1]) return;
    long long p = i * g.st[0] + j * g.st[1];
    long long sz = g.st[2];
    int Nz = g.N[2];
    auto zb = [&](int k) -> FT {
        // the buoyancy model is a template parameter: with a run-time switch in here the 16 loads of a batch were no
        // longer issued together (hydrostatic 0.20 -> 0.34 ms per step)
        if (BMODE == BUOY_NONE) return FT(0);
        const long long q = p + k * sz;
        FT v = BMODE == BUOY_TRACER ? b.T[q] : BMODE == BUOY_TS ? b.g * (b.alpha * b.T[q] - b.beta * b.S[q])
             : BMODE == BUOY_T ? b.ga * b.T[q] : b.ngb * b.S[q];
        return tilted ? gz * v : v;
    };
    FT above = zb(WRAP ? 1 : Nz + 1), acc = FT(0);
    for (int kt = Nz; kt >= 1; kt -= HU) {
        FT v[HU];
#pragma unroll
        for (int u = 0; u < HU; ++u) v[u] = kt - u >= 1 ? zb(kt - u) : FT(0);
#pragma unroll
        for (int u = 0; u < HU; ++u) {
            int k = kt - u;
            if (k >= 1) {
                FT t = (FT(0.5) * (v[u] + above)) * spacing(g, 2, OB_F, k + 1);
                acc = k == Nz ? -t : acc - t;
                pHY[p + k * sz] = acc;
                above = v[u];
            }
        }
    }
}
template <class FT>
void launch_hydrostatic_pressure(const GridD<FT>& g, const Buoy<FT>& b, FT gz, FT* pHY, bool periodic_wrap) {
    dim3 blk(32, 2), grd(cdiv(g.N[0], 32), cdiv(g.N[1], 2));
    const bool wrap = periodic_wrap && g.topo[2] == OB_PERIODIC;
#define HY(M)                                                                                              \
    case M:                                                                                                \
        if (wrap) hydrostatic_kernel<FT, true, M><<<grd, blk, 0, stream()>>>(g, b, gz, gz != FT(1), pHY);  \
        else hydrostatic_kernel<FT, false, M><<<grd, blk, 0, stream()>>>(g, b, gz, gz != FT(1), pHY);      \
        break;
    switch (b.mode) { HY(BUOY_TRACER) HY(BUOY_TS) HY(BUOY_T) HY(BUOY_S) default: HY(BUOY_NONE) }
#undef HY
    OB_LAUNCH_CHECK();
}
template void launch_hydrostatic_pressure<float>(const GridD<float>&, const Buoy<float>&, float, float*, bool);
template void launch_hydrostatic_pressure<double>(const GridD<double>&, const Buoy<double>&, double, double*, bool);

// =============================================================================================
// reference parent layout <-> internal layout
// =============================================================================================
template <class FT, bool TO_INTERNAL>
__global__ void convert_kernel(GridD<FT> g, int p0, int p1, int p2, const FT* src, FT* dst) {
    int a = blockIdx.x * blockDim.x + threadIdx.x;
    int b = blockIdx.y * blockDim.y + threadIdx.y;
    int c = blockIdx.z;
    if (a >= p0 || b >= p1 || c >= p2) return;
    long long ip = a + (long long)p0 * (b + (long long)p1 * c);           // parent (reference) index
    long long ii = (a - g.H[0] + g.O[0]) * g.st[0] + (b - g.H[1] + g.O[1]) * g.st[1] +
                   (c - g.H[2] + g.O[2]) * g.st[2];
    if (TO_INTERNAL) dst[ii] = src[ip];
    else dst[ip] = src[ii];
}
template <class FT>
void launch_to_internal(const GridD<FT>& g, const int ps[3], const int loc[3], const FT* parent, FT* base) {
    dim3 blk(64, 4, 1), grd(cdiv(ps[0], 64), cdiv(ps[1], 4), ps[2]);
    convert_kernel<FT, true><<<grd, blk, 0, stream()>>>(g, ps[0], ps[1], ps[2], parent, base);
    OB_LAUNCH_CHECK();
}
template <class FT>
void launch_from_internal(const GridD<FT>& g, const int ps[3], const int loc[3], const FT* base, FT* parent) {
    dim3 blk(64, 4, 1), grd(cdiv(ps[0], 64), cdiv(ps[1], 4), ps[2]);
    convert_kernel<FT, false><<<grd, blk, 0, stream()>>>(g, ps[0], ps[1], ps[2], base, parent);
    OB_LAUNCH_CHECK();
}
template void launch_to_internal<float>(const GridD<float>&, const int[3], const int[3], const float*, float*);
template void launch_to_internal<double>(const GridD<double>&, const int[3], const int[3], const double*, double*);
template void launch_from_internal<float>(const GridD<float>&, const int[3], const int[3], const float*, float*);
template void launch_from_internal<double>(const GridD<double>&, const int[3], const int[3], const double*, double*);

// =============================================================================================
// reductions
// =============================================================================================
__device__ __forceinline__ void block_reduce_store(double s, double s2, double mx, int nan, double* out4) {
    __shared__ double sh[4][32];
    int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    for (int o = 16; o > 0; o >>= 1) {
        s += __shfl_down_sync(0xffffffff, s, o);
        s2 += __shfl_down_sync(0xffffffff, s2, o);
        mx = fmax(mx, __shfl_down_sync(0xffffffff, mx, o));
        nan |= __shfl_down_sync(0xffffffff, nan, o);
    }
    if (lane == 0) { sh[0][wid] = s; sh[1][wid] = s2; sh[2][wid] = mx; sh[3][wid] = nan; }
    __syncthreads();
    if (wid == 0) {
        int nw = (blockDim.x + 31) >> 5;
        s = lane < nw ? sh[0][lane] : 0; s2 = lane < nw ? sh[1][lane] : 0;
        mx = lane < nw ? sh[2][lane] : 0; double nn = lane < nw ? sh[3][lane] : 0;
        for (int o = 16; o > 0; o >>= 1) {
            s += __shfl_down_sync(0xffffffff, s, o);
            s2 += __shfl_down_sync(0xffffffff, s2, o);
            mx = fmax(mx, __shfl_down_sync(0xffffffff, mx, o));
            nn += __shfl_down_sync(0xffffffff, nn, o);
        }
        if (lane == 0) {
            atomicAdd(out4 + 0, s);
            atomicAdd(out4 + 1, s2);
            atomicMax((unsigned long long*)(out4 + 2), (unsigned long long)__double_as_longlong(mx));
            if (nn > 0) atomicAdd(out4 + 3, 1.0);
        }
    }
}

// calculate_nonlinear_viscosity! (turbulence_closure_utils.jl:35-38) for SmagorinskyLilly: νₑ over the interior
template <class FT>
__global__ void __launch_bounds__(128) smagorinsky_kernel(const __grid_constant__ Phys<FT> P, const Buoy<FT> B, const FT* u,
                                                          const FT* v, const FT* w, FT* nue) {
    const GridD<FT>& g = P.g;
    int i = 1 + blockIdx.x * blockDim.x + threadIdx.x;
    int j = 1 + blockIdx.y * blockDim.y + threadIdx.y;
    int k = 1 + blockIdx.z;
    if (i > g.N[0] || j > g.N[1]) return;
    Pt q;
    q.i[0] = i; q.i[1] = j; q.i[2] = k;
    q.p = i * g.st[0] + j * g.st[1] + k * g.st[2];
    const FT* U[3] = {u, v, w};
    nue[q.p] = smagorinsky_nu(P, B, U, q);
}
// implicit_step! (vertically_implicit_diffusion_solver.jl:153-195) = solve!(field, ::BatchedTridiagonalSolver, field, ...)
// (batched_tridiagonal_solver.jl:91-122) with the coefficient functions ivd_lower_diagonal / ivd_diagonal / ivd_upper_diagonal
// (:27-72) evaluated on the fly for a constant diffusivity: one (i, j) column per thread, in place, k = 1 .. Nz.
// ZFACE: the field lives at z Faces (w): the reference's Face variants of the coefficients.
template <class FT, bool ZFACE>
__global__ void __launch_bounds__(128) ivd_kernel(GridD<FT> g, FT* f, FT* t, FT kappa, FT dt) {
    const int i = 1 + blockIdx.x * blockDim.x + threadIdx.x, j = 1 + blockIdx.y;
    if (i > g.N[0]) return;
    const long long p = i * g.st[0] + j * g.st[1], sz = g.st[2];
    const int Nz = g.N[2];
    auto dzc = [&](int k) { return spacing(g, 2, OB_C, k); };
    auto dzf = [&](int k) { return spacing(g, 2, OB_F, k); };
    auto kdz2 = [&](int kc, int kf) { return kappa / dzc(kc) / dzf(kf); };          // κ_Δz²
    auto upper = [&](int k) -> FT {
        if (ZFACE) return k < 1 ? FT(0) : -dt * kdz2(k, k);
        return k > Nz - 1 ? FT(0) : -dt * kdz2(k, k + 1);
    };
    auto lower = [&](int k) -> FT {
        if (k < 1) return FT(0);
        return ZFACE ? -dt * kdz2(k + 1, k) : -dt * kdz2(k + 1, k + 1);
    };
    auto diag = [&](int k) -> FT { return FT(1) - dt * FT(0) - upper(k) - lower(k - 1); };
    const FT eps10 = 10 * (sizeof(FT) == 4 ? FT(1.1920928955078125e-07) : FT(2.220446049250313e-16));
    FT beta = diag(1);
    FT prev = f[p + sz] / beta;
    f[p + sz] = prev;
    for (int k = 2; k <= Nz; ++k) {
        const FT ck = upper(k - 1), bk = diag(k), ak = lower(k - 1);
        const FT tk = ck / beta;
        t[p + k * sz] = tk;
        beta = bk - ak * tk;
        if (!(fabs(beta) > eps10)) break;
        const FT r = (f[p + k * sz] - ak * prev) / beta;
        f[p + k * sz] = r;
        prev = r;
    }
    FT nxt = f[p + (long long)Nz * sz];
    for (int k = Nz - 1; k >= 1; --k) {
        const FT v = f[p + k * sz] - t[p + (k + 1) * sz] * nxt;
        f[p + k * sz] = v;
        nxt = v;
    }
}
template <class FT>
void launch_implicit_vertical_diffusion(const GridD<FT>& g, FT* field_p0, FT* scratch_p0, FT kappa, FT dt, bool z_face) {
    dim3 blk(64), grd(cdiv(g.N[0], 64), g.N[1]);
    if (z_face) ivd_kernel<FT, true><<<grd, blk, 0, stream()>>>(g, field_p0, scratch_p0, kappa, dt);
    else ivd_kernel<FT, false><<<grd, blk, 0, stream()>>>(g, field_p0, scratch_p0, kappa, dt);
    OB_LAUNCH_CHECK();
}
template void launch_implicit_vertical_diffusion<float>(const GridD<float>&, float*, float*, float, float, bool);
template void launch_implicit_vertical_diffusion<double>(const GridD<double>&, double*, double*, double, double, bool);

// calculate_nonlinear_viscosity! + calculate_nonlinear_tracer_diffusivity! for AnisotropicMinimumDissipation
// (anisotropic_minimum_dissipation.jl:222-251): νₑ and every tracer's κₑ over the interior in one launch
template <class FT>
struct AmdArgs { const FT* u; const FT* v; const FT* w; FT* nue; int ntr; const FT* c[8]; FT* ke[8]; };
template <class FT>
__global__ void __launch_bounds__(128) amd_kernel(const __grid_constant__ Phys<FT> P, const Buoy<FT> B, const AmdArgs<FT> A) {
    const GridD<FT>& g = P.g;
    int i = 1 + blockIdx.x * blockDim.x + threadIdx.x;
    int j = 1 + blockIdx.y * blockDim.y + threadIdx.y;
    int k = 1 + blockIdx.z;
    if (i > g.N[0] || j > g.N[1]) return;
    Pt q;
    q.i[0] = i; q.i[1] = j; q.i[2] = k;
    q.p = i * g.st[0] + j * g.st[1] + k * g.st[2];
    const FT* U[3] = {A.u, A.v, A.w};
    if (g.topo[0] != OB_FLAT && g.topo[1] != OB_FLAT && g.topo[2] != OB_FLAT) {
        FT nu, ka[8];
        amd_cell<FT>(P, B, U, A.ntr, A.c, q, nu, ka);
        A.nue[q.p] = nu;
        for (int t = 0; t < A.ntr; ++t) A.ke[t][q.p] = ka[t];
        return;
    }
    A.nue[q.p] = amd_nu(P, B, U, q);
    for (int t = 0; t < A.ntr; ++t) A.ke[t][q.p] = amd_kappa(P, P.amdCk[t], U, A.c[t], q);
}
template <class FT>
void launch_amd(const Phys<FT>& P, const Buoy<FT>& B, const FT* u, const FT* v, const FT* w, FT* nue, int ntr,
                const FT* const* c, FT* const* ke) {
    const GridD<FT>& g = P.g;
    AmdArgs<FT> A;
    A.u = u; A.v = v; A.w = w; A.nue = nue; A.ntr = ntr;
    for (int t = 0; t < ntr; ++t) { A.c[t] = c[t]; A.ke[t] = ke[t]; }
    dim3 blk(32, 4), grd(cdiv(g.N[0], 32), cdiv(g.N[1], 4), g.N[2]);
    amd_kernel<FT><<<grd, blk, 0, stream()>>>(P, B, A);
    OB_LAUNCH_CHECK();
}
template void launch_amd<float>(const Phys<float>&, const Buoy<float>&, const float*, const float*, const float*, float*, int,
                                const float* const*, float* const*);
template void launch_amd<double>(const Phys<double>&, const Buoy<double>&, const double*, const double*, const double*, double*, int,
                                 const double* const*, double* const*);

template <class FT>
void launch_smagorinsky(const Phys<FT>& P, const Buoy<FT>& B, const FT* u, const FT* v, const FT* w, FT* nue) {
    const GridD<FT>& g = P.g;
    dim3 blk(32, 4), grd(cdiv(g.N[0], 32), cdiv(g.N[1], 4), g.N[2]);
    smagorinsky_kernel<FT><<<grd, blk, 0, stream()>>>(P, B, u, v, w, nue);
    OB_LAUNCH_CHECK();
}
template void launch_smagorinsky<float>(const Phys<float>&, const Buoy<float>&, const float*, const float*, const float*, float*);
template void launch_smagorinsky<double>(const Phys<double>&, const Buoy<double>&, const double*, const double*, const double*, double*);

template <class FT>
__global__ void reduce_kernel(GridD<FT> g, const FT* p0, int l0, int l1, int l2, int n0, int n1, int n2, double* out4) {
    long long total = (long long)n0 * n1 * n2;
    double s = 0, s2 = 0, mx = 0;
    int nan = 0;
    for (long long t = blockIdx.x * (long long)blockDim.x + threadIdx.x; t < total;
         t += (long long)gridDim.x * blockDim.x) {
        int i = l0 + (int)(t % n0);
        int j = l1 + (int)((t / n0) % n1);
        int k = l2 + (int)(t / ((long long)n0 * n1));
        double v = (double)p0[i * g.st[0] + j * g.st[1] + k * g.st[2]];
        if (v != v) nan = 1;
        else { s += v; s2 += v * v; mx = fmax(mx, fabs(v)); }
    }
    block_reduce_store(s, s2, mx, nan, out4);
}
template <class FT>
void launch_reduce_box(const GridD<FT>& g, const FT* p0, const int lo[3], const int n[3], double* out4) {
    OB_CUDA(cudaMemsetAsync(out4, 0, 4 * sizeof(double), stream()));
    long long total = (long long)n[0] * n[1] * n[2];
    int blocks = (int)std::min<long long>(148 * 8, (total + 255) / 256);
    reduce_kernel<FT><<<blocks, 256, 0, stream()>>>(g, p0, lo[0], lo[1], lo[2], n[0], n[1], n[2], out4);
    OB_LAUNCH_CHECK();
}
template <class FT>
void launch_reduce(const GridD<FT>& g, const FT* p0, const int n[3], double* out4) {
    const int lo[3] = {1, 1, 1};
    launch_reduce_box<FT>(g, p0, lo, n, out4);
}
template void launch_reduce<float>(const GridD<float>&, const float*, const int[3], double*);
template void launch_reduce<double>(const GridD<double>&, const double*, const int[3], double*);
template void launch_reduce_box<float>(const GridD<float>&, const float*, const int[3], const int[3], double*);
template void launch_reduce_box<double>(const GridD<double>&, const double*, const int[3], const int[3], double*);

template <class FT>
__global__ void maxdiv_kernel(GridD<FT> g, const FT* u, const FT* v, const FT* w, double* out4) {
    long long total = (long long)g.N[0] * g.N[1] * g.N[2];
    double s = 0, s2 = 0, mx = 0;
    int nan = 0;
    for (long long t = blockIdx.x * (long long)blockDim.x + threadIdx.x; t < total;
         t += (long long)gridDim.x * blockDim.x) {
        Pt q;
        q.i[0] = 1 + (int)(t % g.N[0]);
        q.i[1] = 1 + (int)((t / g.N[0]) % g.N[1]);
        q.i[2] = 1 + (int)(t / ((long long)g.N[0] * g.N[1]));
        q.p = q.i[0] * g.st[0] + q.i[1] * g.st[1] + q.i[2] * g.st[2];
        double dv = (double)div_ccc(g, u, v, w, q);
        if (dv != dv) nan = 1;
        else { mx = fmax(mx, fabs(dv)); s += dv; s2 += dv * dv; }
    }
    block_reduce_store(s, s2, mx, nan, out4);
}
template <class FT>
void launch_max_divergence(const GridD<FT>& g, const FT* u, const FT* v, const FT* w, double* out4) {
    OB_CUDA(cudaMemsetAsync(out4, 0, 4 * sizeof(double), stream()));
    long long total = (long long)g.N[0] * g.N[1] * g.N[2];
    int blocks = (int)std::min<long long>(148 * 8, (total + 255) / 256);
    maxdiv_kernel<FT><<<blocks, 256, 0, stream()>>>(g, u, v, w, out4);
    OB_LAUNCH_CHECK();
}
template void launch_max_divergence<float>(const GridD<float>&, const float*, const float*, const float*, double*);
template void launch_max_divergence<double>(const GridD<double>&, const double*, const double*, const double*, double*);

// ---- output path: on-device slicing and averaging (OutputWriters/fetch_output.jl:24-36 with a FieldSlicer; AveragedField /
// mean(field, dims = ...)) so that only what is written leaves the device --------------------------------------------------
template <class FT>
__global__ void slice_kernel(const FT* __restrict__ p0, long long sy, long long sz, int lo0, int lo1, int lo2, int n0, int n1,
                             long long total, FT* __restrict__ out) {
    for (long long t = blockIdx.x * (long long)blockDim.x + threadIdx.x; t < total; t += (long long)gridDim.x * blockDim.x) {
        const int i = (int)(t % n0), j = (int)((t / n0) % n1), k = (int)(t / ((long long)n0 * n1));
        out[t] = p0[(lo0 + i) + (lo1 + j) * sy + (lo2 + k) * sz];
    }
}
template <class FT>
void launch_slice(const GridD<FT>& g, const FT* p0, const int lo[3], const int n[3], FT* out) {
    const long long total = (long long)n[0] * n[1] * n[2];
    if (total <= 0) return;
    const int blocks = (int)std::min<long long>(148 * 16, (total + 255) / 256);
    slice_kernel<FT><<<blocks, 256, 0, stream()>>>(p0, g.st[1], g.st[2], lo[0], lo[1], lo[2], n[0], n[1], total, out);
    OB_LAUNCH_CHECK();
}
template void launch_slice<float>(const GridD<float>&, const float*, const int[3], const int[3], float*);
template void launch_slice<double>(const GridD<double>&, const double*, const int[3], const int[3], double*);

// one block per output element: sums the box of the averaged dimensions in Float64 in a fixed order (thread-strided partial
// sums, then a shared-memory tree), so the result does not depend on scheduling
template <class FT>
__global__ void __launch_bounds__(256) average_kernel(const FT* __restrict__ p0, long long sy, long long sz, int n0, int n1, int n2,
                                                       int a0, int a1, int a2, FT* __restrict__ out) {
    const int m0 = a0 ? 1 : n0, m1 = a1 ? 1 : n1;
    const int o = blockIdx.x;
    const int oi = o % m0, oj = (o / m0) % m1, ok = o / (m0 * m1);
    const int r0 = a0 ? n0 : 1, r1 = a1 ? n1 : 1, r2 = a2 ? n2 : 1;
    const long long cnt = (long long)r0 * r1 * r2;
    double acc = 0;
    for (long long t = threadIdx.x; t < cnt; t += blockDim.x) {
        const int i = (int)(t % r0), j = (int)((t / r0) % r1), k = (int)(t / ((long long)r0 * r1));
        acc += (double)p0[(1 + oi + i) + (1 + oj + j) * sy + (1 + ok + k) * sz];
    }
    __shared__ double sh[256];
    sh[threadIdx.x] = acc;
    __syncthreads();
    for (int s = 128; s > 0; s >>= 1) {
        if ((int)threadIdx.x < s) sh[threadIdx.x] += sh[threadIdx.x + s];
        __syncthreads();
    }
    if (threadIdx.x == 0) out[o] = (FT)(sh[0] / (double)cnt);
}
template <class FT>
void launch_average(const GridD<FT>& g, const FT* p0, const int n[3], const int dims[3], FT* out) {
    const long long outs = (long long)(dims[0] ? 1 : n[0]) * (dims[1] ? 1 : n[1]) * (dims[2] ? 1 : n[2]);
    if (outs <= 0) return;
    if (outs >= (1LL << 31)) throw Error("average: too many output elements");
    average_kernel<FT><<<(int)outs, 256, 0, stream()>>>(p0, g.st[1], g.st[2], n[0], n[1], n[2], dims[0], dims[1], dims[2], out);
    OB_LAUNCH_CHECK();
}
template void launch_average<float>(const GridD<float>&, const float*, const int[3], const int[3], float*);
template void launch_average<double>(const GridD<double>&, const double*, const int[3], const int[3], double*);

}  // namespace ob
