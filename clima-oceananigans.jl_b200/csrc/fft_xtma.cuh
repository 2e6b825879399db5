// fft_xtma.cuh -- persistent, bulk-copy-pipelined backward x pass of the fast FFT Poisson solver (single GPU).
// Included by fft_fast.cu (uses its radix engine).
//
// A tile is T consecutive y rows of one level k of the half spectrum.  They are CONTIGUOUS in memory (T x NXP complex),
// so a tile is staged with 1-D bulk copies (`cp.async.bulk.shared::cluster.global`, SASS UBLKCP) that complete on an
// mbarrier.  A block is persistent and keeps STAGES tiles in flight: while the threads transform tile i the copies of
// tiles i+1 .. i+STAGES-1 are running.
// The first x kernels loaded with ordinary instructions and sat at 24 % occupancy with long-scoreboard (global load
// latency) as the dominant stall (ncu r1h: 156 us / 93 us for 537 MB / 268 MB of compulsory traffic).
#pragma once

namespace tx {
using namespace tmau;     // tma_util.cuh

constexpr int STAGES = 3;      // tiles in flight per block

// ---- backward x: half spectrum -> real line, written into the haloed field (+ periodic x halos) -----------------
template <class FT, int LOG2M>
__global__ void __launch_bounds__(256) x_c2r_tma_kernel(const __grid_constant__ XArgs<FT> A) {
    using CT = typename Cx<FT>::T;
    using P2 = typename Pair<FT>::T;
    using G = Geo<LOG2M>;
    constexpr int M = 1 << LOG2M;
    extern __shared__ __align__(128) unsigned char smem_raw[];
    __shared__ __align__(8) unsigned long long full[STAGES];
    const int T = A.T;
    const unsigned tile_bytes = (unsigned)T * A.NXP * sizeof(CT);
    const size_t stage_stride = ((size_t)tile_bytes + 127) / 128 * 128;
    CT* s = reinterpret_cast<CT*>(smem_raw + STAGES * stage_stride);     // FFT work lines (padded layout)
    CT* stw = s + T * G::LS;
    for (int w = threadIdx.x; w < M; w += blockDim.x) stw[w] = A.twM[w];
    const bool lead = threadIdx.x == 0;
    if (lead) {
        for (int q = 0; q < STAGES; ++q) mbar_init(&full[q], 1);
        mbar_init_fence();
    }
    __syncthreads();
    const int tiles_y = A.Ny / T, ntiles = tiles_y * A.Nz;          // Ny is a multiple of T (checked on the host)
    const int first = blockIdx.x, step = gridDim.x;
    const int mine = first < ntiles ? (ntiles - first + step - 1) / step : 0;
    auto issue = [&](int n) {
        const int tile = first + n * step;
        const int k = tile / tiles_y, j0 = (tile - k * tiles_y) * T;
        unsigned long long* bar = &full[n % STAGES];
        mbar_expect_tx(bar, tile_bytes);
        bulk_load(smem_raw + (n % STAGES) * stage_stride, A.spec + (long long)A.NXP * (j0 + (long long)A.Ny * k), tile_bytes, bar);
    };
    if (lead) for (int n = 0; n < STAGES && n < mine; ++n) issue(n);

    const int tpl = blockDim.x / T, t = threadIdx.x / tpl, l = threadIdx.x - t * tpl;
    CT* const sl = s + t * G::LS;
    const int Nx = A.Nx, H = A.Hx;
    for (int n = 0; n < mine; ++n) {
        const int slot = n % STAGES;
        const int tile = first + n * step;
        const int k = tile / tiles_y, j0 = (tile - k * tiles_y) * T;
        mbar_wait(&full[slot], (n / STAGES) & 1);
        // tangle: Z[k] = E[k] + i O[k], E = (X[k] + conj X[M-k]) / 2, O = conj(w_N^k) (X[k] - conj X[M-k]) / 2
        const CT* row = reinterpret_cast<const CT*>(smem_raw + slot * stage_stride) + t * A.NXP;
        for (int kk = l; kk < M; kk += tpl) {
            CT a = row[kk], b = row[M - kk];
            CT E, D;
            E.x = FT(0.5) * (a.x + b.x); E.y = FT(0.5) * (a.y - b.y);
            D.x = FT(0.5) * (a.x - b.x); D.y = FT(0.5) * (a.y + b.y);
            CT O = cmulc(D, A.twN[kk]);
            CT Z; Z.x = E.x - O.y; Z.y = E.y + O.x;
            sl[G::pos(A.kpos[kk])] = Z;
        }
        __syncthreads();                      // the staged tile is consumed: its buffer can be refilled
        if (lead && n + STAGES < mine) issue(n + STAGES);
        fft_inv<LOG2M>(s, stw, T);
        FT* orow = A.phi_p0 + (j0 + t + 1) * A.st[1] + (k + 1) * A.st[2];      // Julia (0, j, k)
        for (int m = l; m < M; m += tpl) {
            CT z = sl[G::pos(m)];
            P2 r; r.x = z.x * A.scale; r.y = z.y * A.scale;
            const int i = 2 * m + 1;                 // Julia index of the first of the two reals
            *reinterpret_cast<P2*>(orow + i) = r;
            // periodic halos in x (fill_halo_regions_periodic.jl:37-46)
            if (i > Nx - H) orow[i - Nx] = r.x;
            if (i + 1 > Nx - H) orow[i + 1 - Nx] = r.y;
            if (i <= H) orow[i + Nx] = r.x;
            if (i + 1 <= H) orow[i + 1 + Nx] = r.y;
        }
        __syncthreads();                      // work lines are rewritten by the next tile's tangle
    }
}

}  // namespace tx
