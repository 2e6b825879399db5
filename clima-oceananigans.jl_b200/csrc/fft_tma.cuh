// fft_tma.cuh -- persistent, TMA-pipelined y / z passes of the fast FFT Poisson solver (single GPU).
// Included by fft_fast.cu (shares its radix engine: dft_reg, Rad, brev, freq_of_pos).
//
// The first line kernels staged a tile with ordinary loads, synchronised, transformed, synchronised, stored: with
// two blocks per SM the memory system idled while a block computed and vice versa (ncu r1g: 36-40 % of DRAM peak, 24 %
// warps active).  Here a block is persistent and owns a ring of STAGES tile buffers in shared memory:
//   * one thread issues `cp.async.bulk.tensor.3d` loads (SASS UTMALDG) for tile i+1 while all threads transform
//     tile i, and a bulk tensor STORE (UTMASTG) writes tile i back while tile i+1 is transformed; completion of the
//     loads is tracked with one mbarrier per buffer (expect_tx / try_wait.parity), reuse of a buffer with
//     `cp.async.bulk.wait_group.read`;
//   * a tile is TK consecutive kx of one line set: box (2 TK, N, 1) doubles for lines along y, (2 TK, 1, N) along z,
//     i.e. N rows of TK complex numbers (128 bytes for Float64, TK = 8), which is also the shared-memory layout
//     [m][t] -- every 16-byte access of a quarter warp falls in one 128-byte row, so the radix passes are
//     bank-conflict free without padding;
//   * thread -> (line t = tid % TK, butterfly tid / TK): one radix-16 butterfly per thread and pass in registers.
// The half spectrum is padded to NXP = 8 ceil((Nx/2+1)/8) columns; the pad columns hold zeros and are transformed
// like the others.
#pragma once

namespace tl {

using namespace tmau;     // tma_util.cuh

// addressing of a tile (which tensor maps, which coordinates):
//   ADDR_NAT  in place on the natural half spectrum [Nz][Ny][NXP] (single GPU)
// and, for the slab-decomposed solve (y split over R ranks, chunk layout [R][Nz][NyL][KXB], see fft_fast.cu):
//   ADDR_ZF   z lines: load natural, STORE the KXB columns that belong to rank r into rank r's receive buffer
//             (tensor map over PEER memory: the all-to-all transpose is the store phase of the transform);
//   ADDR_ZI   z lines: load from the chunk layout (4-D map), store natural;
//   ADDR_Y    gathered y lines (m = s NyL + yl): load all R chunks of a column block with one 4-D box, transform,
//             store the part that came from rank s back into rank s's buffer (peer memory).
// Tiles of the distributed modes are aligned to chunk boundaries; a tile that sticks out of its chunk is clipped
// by the tensor-map bounds on store and zero-filled on load.
//   ADDR_YS   split y lines: the NyG = R NyL point transform is done as an R-point butterfly across the chunks (separate
//             elementwise kernel, fft_fast.cu: ysplit_kernel) and NyL-point lines INSIDE each chunk (this kernel, in place on
//             the chunk buffer, tiles of 8 columns with 128-byte rows instead of the 32-byte rows 2048-point lines allow);
//             other index o = z R + r (z-major, so that a block of z levels is a contiguous range of o and the three passes
//             of the split transform can be pipelined per z block with the bulk copies), eigenvalue table lamL[r][m]
//             (frequency r + R freq(m)).
enum { ADDR_NAT = 0, ADDR_ZF = 1, ADDR_ZI = 2, ADDR_Y = 3, ADDR_YS = 4 };
template <class FT>
struct TArgs {
    CUtensorMap tm;                 // ADDR_NAT / ZF load, ZI store base..., view as reals: dims (2 NXP, Ny, Nz)
    CUtensorMap tm4;                // ADDR_ZI / ADDR_Y: 4-D view of the local chunk buffer (2 KXB, NyL, Nz, R)
    CUtensorMap tmr[8];             // per-rank 3-D chunk views (peer buffers, or chunk r of the local spectrum)
    int addr, R, KXB, tpc, NyL, kx_base, NXP, Nz;
    int r_only;                     // ADDR_ZF: >= 0 restricts the launch to the tiles of destination chunk r_only (nkx = tpc)
    int o_first;                    // first value of the other index handled by this launch (split launches)
    int line_is_y;                  // 1: lines along y, other = z ; 0: lines along z, other = y
    int nkx, nOther;                // tiles: nkx = NXP / TK columns blocks x nOther lines sets
    const typename Cx<FT>::T* tw;   // exp(-2 pi i t / N)
    FT scale;
    const double* lamx;             // natural kx
    const double* lamL;             // along the line, position order
    const double* lamO;             // along the other dimension, its storage order
};

// one forward (DIF) radix-R pass on the [m][t] tile; S = stride of the butterfly inputs
template <int R, int LOG2N, int TK, class CT>
__device__ __forceinline__ void pass_fwd_t(CT* s, const CT* tw, int S) {
    constexpr int N = 1 << LOG2N, nb = N / R, LB = ilog2c(R);
    const int m = R * S;
    for (int w = threadIdx.x; w < TK * nb; w += blockDim.x) {
        const int t = w % TK, b = w / TK;
        const int blk = b / S, j = b - blk * S;
        CT* col = s + t;
        const int base = blk * m + j;
        CT x[R];
#pragma unroll
        for (int q = 0; q < R; ++q) x[q] = col[(base + q * S) * TK];
        dft_reg<R, false>(x);
        const int tstep = j * (N / m);
#pragma unroll
        for (int sidx = 0; sidx < R; ++sidx) {
            CT v = x[brev(sidx, LB)];
            if (sidx > 0 && S > 1) v = cmul(v, tw[tstep * sidx]);
            col[(base + sidx * S) * TK] = v;
        }
    }
}
template <int R, int LOG2N, int TK, class CT, class FT>
__device__ __forceinline__ void pass_inv_t(CT* s, const CT* tw, int S, FT scale) {
    constexpr int N = 1 << LOG2N, nb = N / R, LB = ilog2c(R);
    const int m = R * S;
    for (int w = threadIdx.x; w < TK * nb; w += blockDim.x) {
        const int t = w % TK, b = w / TK;
        const int blk = b / S, j = b - blk * S;
        CT* col = s + t;
        const int base = blk * m + j;
        const int tstep = j * (N / m);
        CT x[R];
#pragma unroll
        for (int sidx = 0; sidx < R; ++sidx) {
            CT v = col[(base + sidx * S) * TK];
            if (sidx > 0 && S > 1) v = cmulc(v, tw[tstep * sidx]);
            x[sidx] = v;
        }
        dft_reg<R, true>(x);
#pragma unroll
        for (int q = 0; q < R; ++q) {
            CT v = x[brev(q, LB)];
            v.x *= scale; v.y *= scale;          // scale = 1 except in the last backward pass
            col[(base + q * S) * TK] = v;
        }
    }
}

template <class FT, int LOG2N, int MODE, int TK, int STAGES>
__global__ void __launch_bounds__(256) line_tma_kernel(const __grid_constant__ TArgs<FT> A) {
    using CT = typename Cx<FT>::T;
    using R = Rad<LOG2N>;
    constexpr int N = 1 << LOG2N;
    constexpr unsigned TILE_BYTES = (unsigned)N * TK * sizeof(CT);
    extern __shared__ __align__(128) unsigned char smem_raw[];
    __shared__ __align__(8) unsigned long long full[STAGES];
    CT* stw = reinterpret_cast<CT*>(smem_raw + (size_t)STAGES * TILE_BYTES);
    auto buf = [&](int slot) { return reinterpret_cast<CT*>(smem_raw + (size_t)slot * TILE_BYTES); };
    for (int w = threadIdx.x; w < N; w += blockDim.x) stw[w] = A.tw[w];
    const bool lead = threadIdx.x == 0;
    if (lead) {
        for (int q = 0; q < STAGES; ++q) mbar_init(&full[q], 1);
        mbar_init_fence();
    }
    __syncthreads();

    const int ntiles = A.nkx * A.nOther;
    const int first = blockIdx.x, step = gridDim.x;
    const int mine = first < ntiles ? (ntiles - first + step - 1) / step : 0;
    // tile -> (column block kxb [in units of TK columns; within chunk r for the distributed modes], other index o,
    // chunk r); kx0 = first global kx of the tile
    auto coords = [&](int n, int& kxb, int& o, int& r, int& kx0) {
        const int tile = first + n * step;
        o = tile / A.nkx; kxb = tile - o * A.nkx;
        o += A.o_first;
        r = 0;
        if (A.addr == ADDR_ZF && A.r_only >= 0) { r = A.r_only; kx0 = r * A.KXB + TK * kxb; }
        else if (A.addr == ADDR_ZF || A.addr == ADDR_ZI) { r = kxb / A.tpc; kxb -= r * A.tpc; kx0 = r * A.KXB + TK * kxb; }
        else {
            kx0 = A.kx_base + TK * kxb;
            if (A.addr == ADDR_YS) r = o % A.R;
        }
    };
    auto issue_load = [&](int n) {
        int kxb, o, r, kx0;
        coords(n, kxb, o, r, kx0);
        unsigned long long* bar = &full[n % STAGES];
        mbar_expect_tx(bar, TILE_BYTES);
        void* dst = buf(n % STAGES);
        if (A.addr == ADDR_NAT) {
            // a box holds at most 256 rows: lines of 512 points are staged as two boxes
            constexpr int ROWS = N > 256 ? 256 : N;
#pragma unroll
            for (int b = 0; b < N / ROWS; ++b)
                tma_load_3d(reinterpret_cast<CT*>(dst) + (size_t)b * ROWS * TK, &A.tm, 2 * kx0, A.line_is_y ? b * ROWS : o,
                            A.line_is_y ? o : b * ROWS, bar);
        }
        else if (A.addr == ADDR_ZF) tma_load_3d(dst, &A.tm, 2 * kx0, o, 0, bar);
        else if (A.addr == ADDR_ZI) tma_load_4d(dst, &A.tm4, 2 * TK * kxb, o, 0, r, bar);
        else if (A.addr == ADDR_YS) tma_load_4d(dst, &A.tm4, 2 * TK * kxb, 0, o / A.R, r, bar);
        else tma_load_4d(dst, &A.tm4, 2 * TK * kxb, 0, o, 0, bar);
    };
    if (lead && mine > 0) issue_load(0);
    (void)0;

    for (int n = 0; n < mine; ++n) {
        const int slot = n % STAGES;
        if (lead && n + 1 < mine) {
            // buffer (n+1) % STAGES was stored from STAGES-1 tiles ago: allow the STAGES-2 most recent stores in flight
            bulk_wait_read<STAGES - 2>();
            issue_load(n + 1);
        }
        mbar_wait(&full[slot], (n / STAGES) & 1);
        CT* s = buf(slot);
        int kxb, o, r, kx0;
        coords(n, kxb, o, r, kx0);

        if constexpr (MODE == LM_FWD) {
            pass_fwd_t<R::R1, LOG2N, TK>(s, stw, N / R::R1);
            if constexpr (R::R2 > 1) { __syncthreads(); pass_fwd_t<R::R2, LOG2N, TK>(s, stw, N / (R::R1 * R::R2)); }
            if constexpr (R::R3 > 1) { __syncthreads(); pass_fwd_t<R::R3, LOG2N, TK>(s, stw, 1); }
        } else if constexpr (MODE == LM_INV) {
            constexpr bool l3 = R::R3 > 1, l2 = R::R2 > 1;
            if constexpr (l3) { pass_inv_t<R::R3, LOG2N, TK>(s, stw, 1, FT(1)); __syncthreads(); }
            if constexpr (l2) { pass_inv_t<R::R2, LOG2N, TK>(s, stw, N / (R::R1 * R::R2), FT(1)); __syncthreads(); }
            pass_inv_t<R::R1, LOG2N, TK>(s, stw, N / R::R1, A.scale);
        } else {
            constexpr int RLAST = R::R3 > 1 ? R::R3 : (R::R2 > 1 ? R::R2 : R::R1);
            if constexpr (R::R2 > 1) { pass_fwd_t<R::R1, LOG2N, TK>(s, stw, N / R::R1); __syncthreads(); }
            if constexpr (R::R3 > 1) { pass_fwd_t<R::R2, LOG2N, TK>(s, stw, N / (R::R1 * R::R2)); __syncthreads(); }
            // last forward pass (stride 1, no twiddles), eigenvalue divide, first backward pass, in registers:
            // phi_hat = -b_hat / (lx + ly + lz), zero mode = 0 (fft_based_poisson_solver.jl:106-111)
            constexpr int nb = N / RLAST, LB = ilog2c(RLAST);
            constexpr bool single = R::R2 == 1;        // one-pass transform: the scale belongs here
            for (int w = threadIdx.x; w < TK * nb; w += blockDim.x) {
                const int t = w % TK, blk = w / TK, base = blk * RLAST;
                CT* col = s + t;
                CT x[RLAST], y[RLAST];
#pragma unroll
                for (int q = 0; q < RLAST; ++q) x[q] = col[(base + q) * TK];
                dft_reg<RLAST, false>(x);
                const int kx = min(kx0 + t, A.NXP - 1);       // columns clipped out of a chunk carry zeros
                const int oz = A.addr == ADDR_YS ? o / A.R : o;
                const double* lamLr = A.addr == ADDR_YS ? A.lamL + r * N : A.lamL;
                const double lO = A.lamO ? A.lamO[oz] : 0.0;
                const double lxo = A.line_is_y ? A.lamx[kx] : (A.lamx[kx] + lO);
#pragma unroll
                for (int sidx = 0; sidx < RLAST; ++sidx) {
                    const int m = base + sidx;
                    const double lL = lamLr[m];
                    const double lam = A.line_is_y ? ((lxo + lL) + lO) : (lxo + lL);
                    const CT v = x[brev(sidx, LB)];
                    const double r = (kx == 0 && m == 0 && o == 0) ? 0.0 : -rcp_full(lam);
                    y[sidx].x = (FT)((double)v.x * r); y[sidx].y = (FT)((double)v.y * r);
                }
                dft_reg<RLAST, true>(y);
#pragma unroll
                for (int q = 0; q < RLAST; ++q) {
                    CT v = y[brev(q, LB)];
                    if (single) { v.x *= A.scale; v.y *= A.scale; }
                    col[(base + q) * TK] = v;
                }
            }
            if constexpr (R::R3 > 1) { __syncthreads(); pass_inv_t<R::R2, LOG2N, TK>(s, stw, N / (R::R1 * R::R2), FT(1)); }
            if constexpr (R::R2 > 1) { __syncthreads(); pass_inv_t<R::R1, LOG2N, TK>(s, stw, N / R::R1, A.scale); }
        }
        fence_async_smem();           // generic-proxy writes of the tile -> visible to the bulk store
        __syncthreads();
        if (lead) {
            if (A.addr == ADDR_NAT) {
                constexpr int ROWS = N > 256 ? 256 : N;
#pragma unroll
                for (int b = 0; b < N / ROWS; ++b)
                    tma_store_3d(&A.tm, 2 * kx0, A.line_is_y ? b * ROWS : o, A.line_is_y ? o : b * ROWS, s + (size_t)b * ROWS * TK);
            }
            else if (A.addr == ADDR_ZF || A.addr == ADDR_ZI) tma_store_3d(&A.tmr[r], 2 * TK * kxb, o, 0, s);
            else if (A.addr == ADDR_YS) tma_store_3d(&A.tmr[r], 2 * TK * kxb, 0, o / A.R, s);
            else for (int q = 0; q < A.R; ++q) tma_store_3d(&A.tmr[q], 2 * TK * kxb, 0, o, s + (size_t)q * A.NyL * TK);
            bulk_commit();
        }
    }
    if (lead) bulk_wait_all();        // shared memory must outlive the last stores; peer writes are complete at exit
}

}  // namespace tl
