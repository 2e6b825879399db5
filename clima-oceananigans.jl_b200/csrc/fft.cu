// fft.cu -- batched 1-D transforms in shared memory, the FFT-based Poisson solver, the
// Fourier-tridiagonal solver and the batched Thomas kernel.  sm_100a, FP64/FP32.
//
// Reference: Solvers/fft_based_poisson_solver.jl:93-125, poisson_eigenvalues.jl:8-31,
// discrete_transforms.jl:25-33 (normalisation), fourier_tridiagonal_poisson_solver.jl:16-123,
// batched_tridiagonal_solver.jl:91-122.  The reference calls FFTW/cuFFT; here the transforms
// are hand-written:
//   * power-of-two Periodic dims: in-place radix-2 butterflies in shared memory.  Forward is
//     decimation-in-frequency (natural in, bit-reversed out), backward is decimation-in-time
//     (bit-reversed in, natural out), so NO reordering pass exists anywhere: spectral data
//     simply lives in bit-reversed order along such a dimension, and the eigenvalue tables are
//     uploaded in that same order.
//   * Bounded dims (DCT-II / DCT-III with the FFTW REDFT10 / REDFT01/(2N) conventions): Makhoul's algorithm -- the
//     even / odd permutation of the line (index_permutations.jl:18-94 does the same for the reference's GPU transforms,
//     discrete_transforms.jl:140-183) folded into the global load / store, one complex FFT of the same length, and a
//     pairwise (k, n-k) twiddle that also separates the transforms of the real and the imaginary part of the line.
//     Power-of-two lengths keep the spectrum in bit-reversed positions like the Periodic ones.
//   * non-power-of-two lengths (Periodic, or the FFT inside a Bounded transform): Bluestein's chirp-z algorithm on the
//     same shared-memory butterflies with M = the power of two >= 2n - 1; spectral order natural.
//   * lengths whose M does not fit shared memory (n > 2048), n = 1 and OB200_DIRECT_TRANSFORMS=1: direct O(n^2)
//     evaluation from an exact twiddle table (the round-1 path, kept as the cross-check of the fast ones).
// A block transforms T lines that are adjacent along the contiguous (x) direction so that
// every global access is a run of T consecutive complex numbers.
#include "internal.h"
#include <vector>
#include <cmath>
#include <algorithm>

namespace ob {

template <class FT> struct Cx;
template <> struct Cx<float> { using T = float2; };
template <> struct Cx<double> { using T = double2; };

enum { TK_POW2 = 0, TK_DFT = 1, TK_DCT = 2, TK_DCT_POW2 = 3, TK_BLUE = 4, TK_DCT_BLUE = 5 };
enum { MODE_FWD = 0, MODE_INV = 1, MODE_FWD_DIV_INV = 2 };

template <class FT>
struct FftArgs {
    typename Cx<FT>::T* data;
    int n, log2n;
    long long stride;              // between consecutive points of a line (complex elements)
    int nA, nB;
    long long strideA, strideB;    // between adjacent lines
    int T;                         // lines per block (adjacent along A)
    int kind;
    const typename Cx<FT>::T* tw;  // POW2: n/2 entries exp(-2 pi i k/n); DFT: n entries; DCT: 4n cos (x only);
                                   // DCT_POW2: n/2 FFT twiddles + n exp(-i pi k/(2n)); BLUE: M/2 FFT twiddles + n chirp
                                   // exp(-i pi k^2/n); DCT_BLUE: the same + n exp(-i pi k/(2n))
    int M, log2M;                  // Bluestein: convolution length
    const typename Cx<FT>::T* bhat;// Bluestein: FFT_M of the conjugate chirp / M, in bit-reversed positions (global memory)
    FT scale;                      // applied after the inverse transform (1/n, or 1/(2n) for DCT)
    // eigenvalue divide (MODE_FWD_DIV_INV): lam[dim] in storage order, dims of (line, A, B)
    const double* lam[3];
    int dimL, dimA, dimB;
    // optional fused output of the real part into a haloed field (last inverse pass)
    FT* phi_p0;
    long long phi_st[3];
    int pad;
};

template <class CT> __device__ __forceinline__ CT cmul(CT a, CT b) {
    CT r;
    r.x = a.x * b.x - a.y * b.y;
    r.y = a.x * b.y + a.y * b.x;
    return r;
}
template <class CT> __device__ __forceinline__ CT cmulc(CT a, CT b) {   // a * conj(b)
    CT r;
    r.x = a.x * b.x + a.y * b.y;
    r.y = a.y * b.x - a.x * b.y;
    return r;
}

// in-place radix-2 on T lines held in shared memory (line stride LS)
template <class FT, bool INVERSE>
__device__ __forceinline__ void pow2_fft_smem(typename Cx<FT>::T* s, const typename Cx<FT>::T* tw, int n,
                                              int log2n, int T, int LS) {
    using CT = typename Cx<FT>::T;
    int half = n >> 1;
    int total = T * half;
    if (!INVERSE) {                       // DIF: h = n/2 ... 1
        for (int st = 0; st < log2n; ++st) {
            int h = half >> st;
            int tstep = 1 << st;          // twiddle index step: n/(2h)
            const int lh = log2n - 1 - st;        // h = 2^lh: shifts instead of integer divisions
            for (int w = threadIdx.x; w < total; w += blockDim.x) {
                int t = w >> (log2n - 1), bf = w & (half - 1);
                int r = bf & (h - 1), j = ((bf >> lh) << (lh + 1)) + r;
                CT* x = s + t * LS;
                CT a = x[j], b = x[j + h];
                CT su, di;
                su.x = a.x + b.x; su.y = a.y + b.y;
                di.x = a.x - b.x; di.y = a.y - b.y;
                x[j] = su;
                x[j + h] = cmul(di, tw[r * tstep]);
            }
            __syncthreads();
        }
    } else {                              // DIT with conjugate twiddles: h = 1 ... n/2
        for (int st = log2n - 1; st >= 0; --st) {
            int h = half >> st;
            int tstep = 1 << st;
            const int lh = log2n - 1 - st;
            for (int w = threadIdx.x; w < total; w += blockDim.x) {
                int t = w >> (log2n - 1), bf = w & (half - 1);
                int r = bf & (h - 1), j = ((bf >> lh) << (lh + 1)) + r;
                CT* x = s + t * LS;
                CT a = x[j], b = cmulc(x[j + h], tw[r * tstep]);
                CT su, di;
                su.x = a.x + b.x; su.y = a.y + b.y;
                di.x = a.x - b.x; di.y = a.y - b.y;
                x[j] = su;
                x[j + h] = di;
            }
            __syncthreads();
        }
    }
}

// ---- Makhoul DCT-II / DCT-III around a complex FFT of the same length ------------------------------------------------------
// position of element m of the line in the transform's input: evens ascending, then odds descending
__device__ __forceinline__ int dct_perm(int m, int n) { return (m & 1) ? n - 1 - (m >> 1) : (m >> 1); }
template <bool BR> __device__ __forceinline__ int spos(int k, int log2n) {
    return BR ? (int)(__brev((unsigned)k) >> (32 - log2n)) : k;
}
// after the FFT V of the permuted line: Y_k = 2 Re(w_k V_k) separately for the real and the imaginary part of the line,
// i.e. with A = w_k V_k, B = w_k conj(V_{n-k}): Y_k = (Re A + Re B) + i (Im A - Im B); in place on the pair (k, n-k)
template <class FT, bool BR>
__device__ __forceinline__ void dct_post(typename Cx<FT>::T* s, const typename Cx<FT>::T* wk, int n, int log2n, int T, int LS) {
    using CT = typename Cx<FT>::T;
    const int np = n / 2 + 1, total = T * np;
    for (int w = threadIdx.x; w < total; w += blockDim.x) {
        const int t = w / np, k = w - t * np, m = (n - k) % n;
        if (m < k) continue;
        CT* x = s + t * LS;
        const int pk = spos<BR>(k, log2n), pm = spos<BR>(m, log2n);
        const CT Vk = x[pk], Vm = x[pm];
        CT A = cmul(wk[k], Vk), B = cmulc(wk[k], Vm), Y;      // w conj(V) = conj(conj(w) V); cmulc(a, b) = a conj(b)
        Y.x = A.x + B.x; Y.y = A.y - B.y;
        x[pk] = Y;
        if (m != k) {
            A = cmul(wk[m], Vm); B = cmulc(wk[m], Vk);
            Y.x = A.x + B.x; Y.y = A.y - B.y;
            x[pm] = Y;
        }
    }
    __syncthreads();
}
// before the inverse FFT: R_k = conj(w_k) [(Re Y_k + Im Y_{n-k}) + i (Im Y_k - Re Y_{n-k})], Y_n := 0; the unnormalised
// inverse FFT of R is 2n x the permuted line, which is REDFT01's scaling
template <class FT, bool BR>
__device__ __forceinline__ void dct_pre(typename Cx<FT>::T* s, const typename Cx<FT>::T* wk, int n, int log2n, int T, int LS) {
    using CT = typename Cx<FT>::T;
    const int np = n / 2 + 1, total = T * np;
    for (int w = threadIdx.x; w < total; w += blockDim.x) {
        const int t = w / np, k = w - t * np, m = (n - k) % n;
        if (m < k) continue;
        CT* x = s + t * LS;
        const int pk = spos<BR>(k, log2n), pm = spos<BR>(m, log2n);
        const CT Yk = x[pk];
        CT Ym = x[pm], Z;
        if (k == 0) { Ym.x = 0; Ym.y = 0; }
        Z.x = Yk.x + Ym.y; Z.y = Yk.y - Ym.x;
        x[pk] = cmulc(Z, wk[k]);
        if (m != k) {
            Z.x = Ym.x + Yk.y; Z.y = Ym.y - Yk.x;
            x[pm] = cmulc(Z, wk[m]);
        }
    }
    __syncthreads();
}

// ---- Bluestein: DFT of any length n as a circular convolution of length M = 2^log2M >= 2n - 1 ---------------------------------
// X_k = c_k sum_j (x_j c_j) conj(c_{k-j}), c_m = exp(-i pi m^2 / n).  INVERSE: the unnormalised inverse DFT as
// conj(DFT(conj(x))).  Natural order in and out, in place in the first n entries of each line (LS >= M).
template <class FT, bool INVERSE>
__device__ __forceinline__ void blue_dft(typename Cx<FT>::T* s, const typename Cx<FT>::T* twM, const typename Cx<FT>::T* chirp,
                                         const typename Cx<FT>::T* __restrict__ bhat, int n, int M, int log2M, int T, int LS) {
    using CT = typename Cx<FT>::T;
    const int total = T * M;
    for (int w = threadIdx.x; w < total; w += blockDim.x) {
        const int t = w / M, j = w - t * M;
        CT v;
        v.x = 0; v.y = 0;
        if (j < n) {
            v = s[t * LS + j];
            if (INVERSE) v.y = -v.y;
            v = cmul(v, chirp[j]);
        }
        s[t * LS + j] = v;
    }
    __syncthreads();
    pow2_fft_smem<FT, false>(s, twM, M, log2M, T, LS);
    for (int w = threadIdx.x; w < total; w += blockDim.x) {
        const int t = w / M, j = w - t * M;
        s[t * LS + j] = cmul(s[t * LS + j], bhat[j]);
    }
    __syncthreads();
    pow2_fft_smem<FT, true>(s, twM, M, log2M, T, LS);
    const int tn = T * n;
    for (int w = threadIdx.x; w < tn; w += blockDim.x) {
        const int t = w / n, j = w - t * n;
        CT v = cmul(s[t * LS + j], chirp[j]);
        if (INVERSE) v.y = -v.y;
        s[t * LS + j] = v;
    }
    __syncthreads();
}

// direct O(n^2) transforms: s (input) -> o (output), both in shared memory
template <class FT, bool INVERSE>
__device__ __forceinline__ void direct_smem(typename Cx<FT>::T* s, typename Cx<FT>::T* o,
                                            const typename Cx<FT>::T* tw, int n, int T, int LS, int kind) {
    using CT = typename Cx<FT>::T;
    int total = T * n;
    for (int w = threadIdx.x; w < total; w += blockDim.x) {
        int t = w / n, k = w - t * n;
        const CT* x = s + t * LS;
        CT acc;
        acc.x = 0; acc.y = 0;
        if (kind == TK_DFT) {
            int idx = 0;
            for (int j = 0; j < n; ++j) {
                CT tv = tw[idx];
                CT v = INVERSE ? cmulc(x[j], tv) : cmul(x[j], tv);
                acc.x += v.x; acc.y += v.y;
                idx += k;
                if (idx >= n) idx -= n;
            }
        } else if (!INVERSE) {            // REDFT10: Y_k = 2 sum_j x_j cos(pi (2j+1) k / (2n))
            int n4 = 4 * n, idx = k % n4, step = (2 * k) % n4;
            for (int j = 0; j < n; ++j) {
                FT c = tw[idx].x;
                acc.x += x[j].x * c; acc.y += x[j].y * c;
                idx += step;
                if (idx >= n4) idx -= n4;
            }
            acc.x *= 2; acc.y *= 2;
        } else {                          // REDFT01: x_j = X_0 + 2 sum_{k>=1} X_k cos(pi (2j+1) k / (2n))
            int n4 = 4 * n, step = (2 * k + 1) % n4, idx = step;
            for (int m = 1; m < n; ++m) {
                FT c = tw[idx].x;
                acc.x += x[m].x * c; acc.y += x[m].y * c;
                idx += step;
                if (idx >= n4) idx -= n4;
            }
            acc.x = x[0].x + 2 * acc.x; acc.y = x[0].y + 2 * acc.y;
        }
        o[t * LS + k] = acc;
    }
    __syncthreads();
}

template <class FT, int MODE>
__global__ void fft_lines_kernel(FftArgs<FT> A) {
    using CT = typename Cx<FT>::T;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    CT* s = reinterpret_cast<CT*>(smem_raw);
    const int n = A.n, T = A.T, kind = A.kind;
    const bool blue = kind == TK_BLUE || kind == TK_DCT_BLUE, fdct = kind == TK_DCT_POW2 || kind == TK_DCT_BLUE;
    const bool direct = kind == TK_DFT || kind == TK_DCT;
    const int LS = (blue ? A.M : n) + A.pad;
    CT* s2 = s + T * LS;                                  // second buffer (direct kinds only)
    CT* stw = direct ? s2 + T * LS : s2;                  // twiddle copy
    const int nfft = blue ? A.M / 2 : n / 2;              // butterflies' twiddles come first in the fast kinds' tables
    const int ntw = kind == TK_POW2 ? n / 2 : kind == TK_DFT ? n : kind == TK_DCT ? 4 * n
                  : kind == TK_DCT_POW2 ? n / 2 + n : kind == TK_BLUE ? A.M / 2 + n : A.M / 2 + 2 * n;
    for (int w = threadIdx.x; w < ntw; w += blockDim.x) stw[w] = A.tw[w];
    const CT* chirp = stw + nfft;                         // Bluestein kinds
    const CT* wk = stw + nfft + (blue ? n : 0);           // Makhoul kinds

    int a0 = blockIdx.x * T, b = blockIdx.y;
    int nl = min(T, A.nA - a0);                           // lines in this block
    long long base = a0 * A.strideA + b * A.strideB;
    int total = nl * n;
    // Makhoul: the even / odd permutation is applied where the line is in physical space -- on the load before a forward
    // transform, on the store after an inverse one
    const bool perm_in = fdct && MODE != MODE_INV, perm_out = fdct && MODE != MODE_FWD;
    // load: consecutive threads take consecutive memory
    if (A.stride == 1) {
        for (int w = threadIdx.x; w < total; w += blockDim.x) {
            int t = w / n, m = w - t * n;
            s[t * LS + (perm_in ? dct_perm(m, n) : m)] = A.data[base + t * A.strideA + m];
        }
    } else {
        for (int w = threadIdx.x; w < total; w += blockDim.x) {
            int m = w / nl, t = w - m * nl;
            s[t * LS + (perm_in ? dct_perm(m, n) : m)] = A.data[base + t * A.strideA + m * A.stride];
        }
    }
    __syncthreads();

    CT* cur = s;
    if (MODE == MODE_FWD || MODE == MODE_FWD_DIV_INV) {
        if (kind == TK_POW2) pow2_fft_smem<FT, false>(s, stw, n, A.log2n, nl, LS);
        else if (kind == TK_DCT_POW2) {
            pow2_fft_smem<FT, false>(s, stw, n, A.log2n, nl, LS);
            dct_post<FT, true>(s, wk, n, A.log2n, nl, LS);
        } else if (kind == TK_BLUE) blue_dft<FT, false>(s, stw, chirp, A.bhat, n, A.M, A.log2M, nl, LS);
        else if (kind == TK_DCT_BLUE) {
            blue_dft<FT, false>(s, stw, chirp, A.bhat, n, A.M, A.log2M, nl, LS);
            dct_post<FT, false>(s, wk, n, 0, nl, LS);
        } else { direct_smem<FT, false>(s, s2, stw, n, nl, LS, kind); cur = s2; }
    }
    if (MODE == MODE_FWD_DIV_INV) {
        // phi_hat = -b_hat / (lx + ly + lz) ; phi_hat[1,1,1] = 0   (fft_based_poisson_solver.jl:106-111)
        for (int w = threadIdx.x; w < total; w += blockDim.x) {
            int t = w / n, m = w - t * n;
            int id[3];
            id[A.dimL] = m; id[A.dimA] = a0 + t; id[A.dimB] = b;
            double l0 = A.lam[0] ? A.lam[0][id[0]] : 0.0, l1 = A.lam[1] ? A.lam[1][id[1]] : 0.0,
                   l2 = A.lam[2] ? A.lam[2][id[2]] : 0.0;
            double lam = (l0 + l1) + l2;
            CT v = cur[t * LS + m];
            CT r;
            if (id[0] == 0 && id[1] == 0 && id[2] == 0) { r.x = 0; r.y = 0; }
            else { r.x = (FT)(-(double)v.x / lam); r.y = (FT)(-(double)v.y / lam); }
            cur[t * LS + m] = r;
        }
        __syncthreads();
    }
    if (MODE == MODE_INV || MODE == MODE_FWD_DIV_INV) {
        if (kind == TK_POW2) pow2_fft_smem<FT, true>(cur, stw, n, A.log2n, nl, LS);
        else if (kind == TK_DCT_POW2) {
            dct_pre<FT, true>(cur, wk, n, A.log2n, nl, LS);
            pow2_fft_smem<FT, true>(cur, stw, n, A.log2n, nl, LS);
        } else if (kind == TK_BLUE) blue_dft<FT, true>(cur, stw, chirp, A.bhat, n, A.M, A.log2M, nl, LS);
        else if (kind == TK_DCT_BLUE) {
            dct_pre<FT, false>(cur, wk, n, 0, nl, LS);
            blue_dft<FT, true>(cur, stw, chirp, A.bhat, n, A.M, A.log2M, nl, LS);
        } else {
            CT* dst = cur == s ? s2 : s;
            direct_smem<FT, true>(cur, dst, stw, n, nl, LS, kind);
            cur = dst;
        }
    }
    const bool scale = (MODE != MODE_FWD);
    // store
    if (A.phi_p0 != nullptr) {        // fused copy_real_component! into the haloed field
        if (A.stride == 1) {
            for (int w = threadIdx.x; w < total; w += blockDim.x) {
                int t = w / n, m = w - t * n;
                int id[3];
                id[A.dimL] = m; id[A.dimA] = a0 + t; id[A.dimB] = b;
                A.phi_p0[(id[0] + 1) * A.phi_st[0] + (id[1] + 1) * A.phi_st[1] + (id[2] + 1) * A.phi_st[2]] =
                    cur[t * LS + (perm_out ? dct_perm(m, n) : m)].x * A.scale;
            }
        } else {
            for (int w = threadIdx.x; w < total; w += blockDim.x) {
                int m = w / nl, t = w - m * nl;
                int id[3];
                id[A.dimL] = m; id[A.dimA] = a0 + t; id[A.dimB] = b;
                A.phi_p0[(id[0] + 1) * A.phi_st[0] + (id[1] + 1) * A.phi_st[1] + (id[2] + 1) * A.phi_st[2]] =
                    cur[t * LS + (perm_out ? dct_perm(m, n) : m)].x * A.scale;
            }
        }
        return;
    }
    if (A.stride == 1) {
        for (int w = threadIdx.x; w < total; w += blockDim.x) {
            int t = w / n, m = w - t * n;
            CT v = cur[t * LS + (perm_out ? dct_perm(m, n) : m)];
            if (scale) { v.x *= A.scale; v.y *= A.scale; }
            A.data[base + t * A.strideA + m] = v;
        }
    } else {
        for (int w = threadIdx.x; w < total; w += blockDim.x) {
            int m = w / nl, t = w - m * nl;
            CT v = cur[t * LS + (perm_out ? dct_perm(m, n) : m)];
            if (scale) { v.x *= A.scale; v.y *= A.scale; }
            A.data[base + t * A.strideA + m * A.stride] = v;
        }
    }
}

// ---------------------------------------------------------------------------------------------
// batched Thomas: one (i, j) column per thread, coalesced in i (batched_tridiagonal_solver.jl:91-122)
// b (main diagonal) is either a full Nx*Ny*Nz double array or generated on the fly for the
// Fourier-tridiagonal solver (compute_main_diagonals! fourier_tridiagonal_poisson_solver.jl:16-28).
// ---------------------------------------------------------------------------------------------
template <class FT, class VT, bool ONTHEFLY>
__global__ void thomas_kernel(int Nx, int Ny, int Nz, const double* a, const double* bfull, const double* c,
                              const double* lamx, const double* lamy, const double* dzF, const double* dzC,
                              const VT* f, VT* phi, FT* tsc) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    int j = blockIdx.y;
    if (i >= Nx) return;
    long long col = i + (long long)Nx * j, pl = (long long)Nx * Ny;
    double lam = ONTHEFLY ? (lamx[i] + lamy[j]) : 0.0;
    auto diag = [&](int k) -> double {     // k is 1-based
        if (!ONTHEFLY) return bfull[col + (k - 1) * pl];
        // dzF / dzC are indexed by the 1-based Julia index directly
        if (k == 1) return -1 / dzF[2] - dzC[1] * lam;
        if (k == Nz) return -1 / dzF[Nz] - dzC[Nz] * lam;
        return -(1 / dzF[k + 1] + 1 / dzF[k]) - dzC[k] * lam;
    };
    // The reference's pivot guard |beta| > 10 eps is absolute.  For the solver's own columns (ONTHEFLY) beta has units of
    // 1/length and the lowest horizontal mode's last pivot is about lam * H: in Float32 that falls below 10 eps once Lx
    // reaches ~100 km, and the `break` would return a wrong column.  There the guard is relative to the row's diagonal
    // (scale free); the singular mean column is pinned explicitly below.  Caller-supplied coefficients keep the reference's.
    const double eps10 = 10 * (sizeof(FT) == 4 ? 1.1920928955078125e-07 : 2.220446049250313e-16);
    double beta = diag(1);
    VT f1 = f[col];
    VT prev;
    if constexpr (sizeof(VT) == sizeof(FT)) { prev = (VT)((double)f1 / beta); }
    else { prev.x = (FT)((double)f1.x / beta); prev.y = (FT)((double)f1.y / beta); }
    phi[col] = prev;
    for (int k = 2; k <= Nz; ++k) {
        double ck = c[k - 2], bk = diag(k), ak = a[k - 2];
        FT t = (FT)(ck / beta);
        tsc[col + (k - 1) * pl] = t;
        beta = bk - ak * (double)t;
        // The reference leaves phi[k..] at whatever the array held (batched_tridiagonal_solver.jl:104).  For the solver's own
        // columns (ONTHEFLY) that content is defined here -- the right-hand side, as in thomas_half_kernel -- and the singular
        // horizontal-mean column of the Neumann problem is ALWAYS pinned at its last row (its pivot is zero in exact
        // arithmetic, rounding noise otherwise): the constant it leaves open is removed with the mean, and the solution no
        // longer depends on noise / noise or on the solver's history.
        if (!(fabs(beta) > (ONTHEFLY ? eps10 * fabs(bk) : eps10)) || (ONTHEFLY && k == Nz && lam == 0.0)) {
            if (ONTHEFLY)
                for (int q = k; q <= Nz; ++q) phi[col + (q - 1) * pl] = f[col + (q - 1) * pl];
            break;
        }
        VT fk = f[col + (k - 1) * pl];
        VT r;
        if constexpr (sizeof(VT) == sizeof(FT)) { r = (VT)(((double)fk - ak * (double)prev) / beta); }
        else {
            r.x = (FT)(((double)fk.x - ak * (double)prev.x) / beta);
            r.y = (FT)(((double)fk.y - ak * (double)prev.y) / beta);
        }
        phi[col + (k - 1) * pl] = r;
        prev = r;
    }
    VT nxt = phi[col + (long long)(Nz - 1) * pl];
    for (int k = Nz - 1; k >= 1; --k) {
        FT t = tsc[col + k * pl];
        VT v = phi[col + (k - 1) * pl];
        if constexpr (sizeof(VT) == sizeof(FT)) { v -= t * nxt; }
        else { v.x -= t * nxt.x; v.y -= t * nxt.y; }
        phi[col + (k - 1) * pl] = v;
        nxt = v;
    }
}

template <class FT>
void batched_tridiagonal(int Nx, int Ny, int Nz, bool is_complex, const double* a, const double* b,
                         const double* c, const void* rhs, void* phi, FT* scratch) {
    using CT = typename Cx<FT>::T;
    dim3 blk(64), grd(cdiv(Nx, 64), Ny);
    if (is_complex)
        thomas_kernel<FT, CT, false><<<grd, blk, 0, stream()>>>(Nx, Ny, Nz, a, b, c, nullptr, nullptr, nullptr,
                                                                 nullptr, (const CT*)rhs, (CT*)phi, scratch);
    else
        thomas_kernel<FT, FT, false><<<grd, blk, 0, stream()>>>(Nx, Ny, Nz, a, b, c, nullptr, nullptr, nullptr,
                                                                 nullptr, (const FT*)rhs, (FT*)phi, scratch);
    OB_LAUNCH_CHECK();
}
template void batched_tridiagonal<float>(int, int, int, bool, const double*, const double*, const double*,
                                         const void*, void*, float*);
template void batched_tridiagonal<double>(int, int, int, bool, const double*, const double*, const double*,
                                          const void*, void*, double*);

// ---------------------------------------------------------------------------------------------
// mean removal + real copy for the Fourier-tridiagonal solver (…_poisson_solver.jl:93-99)
// ---------------------------------------------------------------------------------------------
// one partial sum per block, each in a fixed order (no atomics: the mean, and with it every bit of the solution, must not
// depend on the order in which blocks happen to finish)
constexpr int MEAN_BLOCKS = 1024;
template <class FT>
__global__ void __launch_bounds__(256) sum_real_kernel(const typename Cx<FT>::T* x, long long n, double* partial) {
    double s = 0;
    for (long long t = blockIdx.x * (long long)blockDim.x + threadIdx.x; t < n; t += (long long)gridDim.x * blockDim.x)
        s += (double)x[t].x;
    __shared__ double sh[256];
    sh[threadIdx.x] = s;
    __syncthreads();
    for (int o = 128; o > 0; o >>= 1) {
        if ((int)threadIdx.x < o) sh[threadIdx.x] += sh[threadIdx.x + o];
        __syncthreads();
    }
    if (threadIdx.x == 0) partial[blockIdx.x] = sh[0];
}
template <class FT>
__global__ void __launch_bounds__(256) sub_mean_copy_kernel(typename Cx<FT>::T* x, int Nx, int Ny, int Nz, const double* partial,
                                                            int nparts, FT* phi_p0, long long s0, long long s1, long long s2) {
    long long n = (long long)Nx * Ny * Nz;
    __shared__ double sh[256];
    {   // every block sums the partials in the same order
        double s = 0;
        for (int q = threadIdx.x; q < nparts; q += blockDim.x) s += partial[q];
        sh[threadIdx.x] = s;
        __syncthreads();
        for (int o = 128; o > 0; o >>= 1) {
            if ((int)threadIdx.x < o) sh[threadIdx.x] += sh[threadIdx.x + o];
            __syncthreads();
        }
    }
    FT mean = (FT)(sh[0] / (double)n);
    for (long long t = blockIdx.x * (long long)blockDim.x + threadIdx.x; t < n; t += (long long)gridDim.x * blockDim.x) {
        int i = (int)(t % Nx), j = (int)((t / Nx) % Ny), k = (int)(t / ((long long)Nx * Ny));
        FT v = x[t].x - mean;
        x[t].x = v; x[t].y = 0;
        phi_p0[(i + 1) * s0 + (j + 1) * s1 + (k + 1) * s2] = v;
    }
}

// ---------------------------------------------------------------------------------------------
// plans
// ---------------------------------------------------------------------------------------------
template <class FT>
struct PoissonPlan {
    using CT = typename Cx<FT>::T;
    int kind;                  // 1 = FFT, 2 = Fourier-tridiagonal
    int N[3], topo[3];
    CT* storage = nullptr;     // Nx*Ny*Nz complex
    CT* source = nullptr;      // tridiagonal: transformed source term
    FT* scratch = nullptr;     // tridiagonal: t
    CT* tw[3] = {nullptr, nullptr, nullptr};
    CT* bhat[3] = {nullptr, nullptr, nullptr};      // Bluestein kinds: transformed conjugate chirp
    int tkind[3], log2n[3], M[3] = {0, 0, 0}, log2M[3] = {0, 0, 0};
    double* lam[3] = {nullptr, nullptr, nullptr};   // storage order
    double* dzF = nullptr;     // device, indexable by Julia index 0..Nz+1 (offset applied)
    double* dzC = nullptr;
    double* lower = nullptr;   // 1/ΔzF(k), k = 2..Nz
    double* msum = nullptr;
    ff::FastPoisson<FT>* fast = nullptr;
    std::vector<void*> owned;
};

static int ilog2(int n) { int l = 0; while ((1 << l) < n) ++l; return l; }
static int bitrev(int x, int bits) { int r = 0; for (int b = 0; b < bits; ++b) if (x & (1 << b)) r |= 1 << (bits - 1 - b); return r; }

template <class T> static T* dev_upload(const std::vector<T>& h, std::vector<void*>& owned) {
    T* d = nullptr;
    OB_CUDA(cudaMalloc(&d, std::max<size_t>(1, h.size()) * sizeof(T)));
    OB_CUDA(cudaMemcpy(d, h.data(), h.size() * sizeof(T), cudaMemcpyHostToDevice));
    owned.push_back(d);
    return d;
}

template <class FT> static void launch_lines(FftArgs<FT>& A, int mode, bool contiguous_lines);

template <class FT>
PoissonPlan<FT>* poisson_plan_create(const GridD<FT>& g, int kind, const double* dzF_host, const double* dzC_host) {
    using CT = typename Cx<FT>::T;
    auto* p = new PoissonPlan<FT>();
    p->kind = kind;
    if (kind == 1 && ff::fast_poisson_supported<FT>(g))
        p->fast = ff::fast_poisson_create<FT>(g);
    if (kind == 2 && ff::fast_ft_supported<FT>(g)) {
        // half-spectrum x / y passes + Thomas sweep on the half spectrum (fft_fast.cu); none of the general path's
        // full-spectrum arrays is needed
        int Nz = g.N[2];
        p->fast = ff::fast_poisson_create<FT>(g);
        std::vector<double> f(dzF_host, dzF_host + Nz + 2), c(dzC_host, dzC_host + Nz + 2);
        p->dzF = dev_upload(f, p->owned);
        p->dzC = dev_upload(c, p->owned);
        ff::fast_poisson_set_tridiagonal<FT>(p->fast, p->dzF, p->dzC);
        for (int d = 0; d < 3; ++d) { p->N[d] = g.N[d]; p->topo[d] = g.topo[d]; }
        return p;
    }
    if (g.topo[0] == OB_COMM || g.topo[1] == OB_COMM || g.topo[2] == OB_COMM) {
        if (!p->fast) {
            delete p;
            throw Error("the slab-decomposed Poisson solver needs Periodic power-of-two x, z and a y decomposition "
                        "(FullyConnected y) with 2, 4 or 8 ranks");
        }
        return p;
    }
    const double PI = 3.14159265358979323846;
    size_t tot = (size_t)g.N[0] * g.N[1] * g.N[2];
    OB_CUDA(cudaMalloc(&p->storage, tot * sizeof(CT)));
    OB_CUDA(cudaMemset(p->storage, 0, tot * sizeof(CT)));
    for (int d = 0; d < 3; ++d) {
        int n = g.N[d];
        p->N[d] = n; p->topo[d] = g.topo[d];
        bool pow2 = n >= 2 && (n & (n - 1)) == 0;
        int M = 1;
        while (M < 2 * n - 1) M <<= 1;
        const bool blue_ok = n >= 2 && M <= 4096;
        int tk;
        if (g.topo[d] == OB_BOUNDED) tk = pow2 ? TK_DCT_POW2 : (blue_ok ? TK_DCT_BLUE : TK_DCT);
        else tk = pow2 ? TK_POW2 : (blue_ok ? TK_BLUE : TK_DFT);
        p->tkind[d] = tk; p->log2n[d] = ilog2(n);
        const bool blue = tk == TK_BLUE || tk == TK_DCT_BLUE;
        if (blue) { p->M[d] = M; p->log2M[d] = ilog2(M); }
        if (g.topo[d] == OB_FLAT || (kind == 2 && d == 2)) {    // not transformed
            if (g.topo[d] == OB_FLAT) {
                std::vector<double> z(n, 0.0);
                p->lam[d] = dev_upload(z, p->owned);
            }
            continue;
        }
        // twiddles, computed in long double and rounded once
        std::vector<CT> tw;
        const long double PIL = 3.14159265358979323846264338327950288L;
        if (tk == TK_POW2 || tk == TK_DFT || tk == TK_DCT) {
            int ntw = tk == TK_POW2 ? n / 2 : (tk == TK_DFT ? n : 4 * n);
            tw.resize(std::max(1, ntw));
            for (int k = 0; k < ntw; ++k) {
                long double ang = tk == TK_DCT ? (long double)PI * k / (2.0L * n) : -2.0L * (long double)PI * k / n;
                tw[k].x = (FT)cosl(ang);
                tw[k].y = tk == TK_DCT ? (FT)0 : (FT)sinl(ang);
            }
        } else {
            // butterflies' twiddles (length n or M), [chirp exp(-i pi k^2 / n)], [Makhoul exp(-i pi k / (2n))]
            const int nf = blue ? M : n;
            auto push = [&](long double ang) { CT c; c.x = (FT)cosl(ang); c.y = (FT)sinl(ang); tw.push_back(c); };
            for (int k = 0; k < nf / 2; ++k) push(-2.0L * PIL * k / nf);
            if (blue)
                for (int k = 0; k < n; ++k) push(-PIL * (long double)(((long long)k * k) % (2LL * n)) / n);
            if (tk != TK_BLUE)
                for (int k = 0; k < n; ++k) push(-PIL * k / (2.0L * n));
            if (blue) {
                // FFT_M of b (b_m = conj(chirp_|m|), |m| < n, wrapped) in long double, divided by M, in the bit-reversed
                // positions the decimation-in-frequency butterflies leave the spectrum in
                std::vector<long double> br(M, 0.0L), bi(M, 0.0L);
                for (int m2 = 0; m2 < n; ++m2) {
                    long double ang = PIL * (long double)(((long long)m2 * m2) % (2LL * n)) / n;
                    br[m2] = cosl(ang); bi[m2] = sinl(ang);
                    if (m2) { br[M - m2] = br[m2]; bi[M - m2] = bi[m2]; }
                }
                const int lg = ilog2(M);
                for (int i = 0; i < M; ++i) { int j = bitrev(i, lg); if (j > i) { std::swap(br[i], br[j]); std::swap(bi[i], bi[j]); } }
                for (int len = 2; len <= M; len <<= 1)
                    for (int i = 0; i < M; i += len)
                        for (int j = 0; j < len / 2; ++j) {
                            long double a = -2.0L * PIL * j / len, wr = cosl(a), wi = sinl(a);
                            int u = i + j, v = u + len / 2;
                            long double tr = br[v] * wr - bi[v] * wi, ti = br[v] * wi + bi[v] * wr;
                            br[v] = br[u] - tr; bi[v] = bi[u] - ti; br[u] += tr; bi[u] += ti;
                        }
                std::vector<CT> bh(M);
                for (int pos = 0; pos < M; ++pos) {
                    int f = bitrev(pos, lg);
                    bh[pos].x = (FT)(br[f] / M); bh[pos].y = (FT)(bi[f] / M);
                }
                p->bhat[d] = dev_upload(bh, p->owned);
            }
        }
        p->tw[d] = dev_upload(tw, p->owned);
        // eigenvalues (poisson_eigenvalues.jl:8-31), Float64, then permuted to storage order
        std::vector<double> lam(n);
        double L = (double)g.L[d];
        for (int i = 0; i < n; ++i) {
            double v = g.topo[d] == OB_PERIODIC ? 2 * sin(i * PI / n) / (L / n) : 2 * sin(i * PI / (2.0 * n)) / (L / n);
            lam[i] = v * v;
        }
        std::vector<double> lp(n);
        for (int i = 0; i < n; ++i) lp[i] = lam[(tk == TK_POW2 || tk == TK_DCT_POW2) ? bitrev(i, p->log2n[d]) : i];
        p->lam[d] = dev_upload(lp, p->owned);
    }
    // (Periodic, Periodic, Bounded) on a regular grid: the half-spectrum x / y passes of fft_fast.cu around a z pass of this
    // file's line kernel (Makhoul DCT, eigenvalue divide, inverse DCT) applied to the half spectrum in place
    if (kind == 1 && !p->fast && g.regular[2] && ff::fast_ft_supported<FT>(g) &&
        (p->tkind[2] == TK_DCT_POW2 || p->tkind[2] == TK_DCT_BLUE)) {
        p->fast = ff::fast_poisson_create<FT>(g);
        ff::fast_poisson_set_zhook<FT>(p->fast, [p]() {
            const ff::FastSpecInfo I = ff::fast_poisson_spec_info<FT>(p->fast);
            FftArgs<FT> A;
            A.data = (CT*)I.spec; A.n = I.Nz; A.log2n = p->log2n[2]; A.stride = (long long)I.NXP * I.Ny;
            A.dimL = 2; A.dimA = 0; A.dimB = 1;
            A.nA = I.NXH; A.nB = I.Ny; A.strideA = 1; A.strideB = I.NXP;
            A.kind = p->tkind[2]; A.tw = p->tw[2]; A.M = p->M[2]; A.log2M = p->log2M[2]; A.bhat = p->bhat[2];
            A.scale = (FT)(1.0 / (2.0 * A.n));
            A.lam[0] = I.lamx; A.lam[1] = I.lamy; A.lam[2] = p->lam[2];
            A.phi_p0 = nullptr;
            launch_lines<FT>(A, MODE_FWD_DIV_INV, false);
        });
    }
    // Bounded y (channels): the same half-spectrum x passes, this file's DCT over the y lines of the half spectrum (forward and
    // backward pass), and for z the Periodic lines of fft_fast.cu, the DCT hook above's twin, or the Thomas sweep
    if (!p->fast && ff::fast_bounded_y_supported<FT>(g) && p->tkind[1] == TK_DCT_POW2 &&
        ((kind == 1 && g.regular[2] && (g.topo[2] == OB_PERIODIC || p->tkind[2] == TK_DCT_POW2 || p->tkind[2] == TK_DCT_BLUE)) ||
         (kind == 2 && g.topo[2] == OB_BOUNDED))) {
        p->fast = ff::fast_poisson_create<FT>(g);
        auto lines = [p](int d, int mode) {
            const ff::FastSpecInfo I = ff::fast_poisson_spec_info<FT>(p->fast);
            FftArgs<FT> A;
            A.data = (CT*)I.spec; A.n = p->N[d]; A.log2n = p->log2n[d];
            A.dimL = d; A.dimA = 0; A.dimB = d == 1 ? 2 : 1;
            A.stride = d == 1 ? (long long)I.NXP : (long long)I.NXP * I.Ny;
            A.nA = I.NXH; A.strideA = 1;
            A.nB = d == 1 ? I.Nz : I.Ny; A.strideB = d == 1 ? (long long)I.NXP * I.Ny : (long long)I.NXP;
            A.kind = p->tkind[d]; A.tw = p->tw[d]; A.M = p->M[d]; A.log2M = p->log2M[d]; A.bhat = p->bhat[d];
            A.scale = (FT)(1.0 / (2.0 * A.n));
            A.lam[0] = I.lamx; A.lam[1] = p->lam[1]; A.lam[2] = p->lam[2];
            A.phi_p0 = nullptr;
            launch_lines<FT>(A, mode, false);
        };
        ff::fast_poisson_set_yhook<FT>(p->fast, [lines](int inverse) { lines(1, inverse ? MODE_INV : MODE_FWD); }, p->lam[1]);
        if (kind == 1 && g.topo[2] == OB_BOUNDED) ff::fast_poisson_set_zhook<FT>(p->fast, [lines]() { lines(2, MODE_FWD_DIV_INV); });
        if (kind == 2) {
            int Nz = g.N[2];
            std::vector<double> f(dzF_host, dzF_host + Nz + 2), c(dzC_host, dzC_host + Nz + 2);
            p->dzF = dev_upload(f, p->owned);
            p->dzC = dev_upload(c, p->owned);
            ff::fast_poisson_set_tridiagonal<FT>(p->fast, p->dzF, p->dzC);
        }
    }
    if (kind == 2) {
        int Nz = g.N[2];
        OB_CUDA(cudaMalloc(&p->source, tot * sizeof(CT)));
        OB_CUDA(cudaMemset(p->source, 0, tot * sizeof(CT)));
        OB_CUDA(cudaMalloc(&p->scratch, tot * sizeof(FT)));
        OB_CUDA(cudaMemset(p->scratch, 0, tot * sizeof(FT)));
        // dzF_host / dzC_host: Nz+2 values for Julia indices 0..Nz+1
        std::vector<double> f(dzF_host, dzF_host + Nz + 2), c(dzC_host, dzC_host + Nz + 2), low(std::max(1, Nz - 1));
        for (int k = 2; k <= Nz; ++k) low[k - 2] = 1 / f[k];
        p->dzF = dev_upload(f, p->owned);
        p->dzC = dev_upload(c, p->owned);
        p->lower = dev_upload(low, p->owned);
        std::vector<double> z(MEAN_BLOCKS, 0.0);
        p->msum = dev_upload(z, p->owned);
    }
    return p;
}
template <class FT> void poisson_plan_destroy(PoissonPlan<FT>* p) {
    if (!p) return;
    ff::fast_poisson_destroy(p->fast);
    cudaFree(p->storage);
    if (p->source) cudaFree(p->source);
    if (p->scratch) cudaFree(p->scratch);
    for (void* q : p->owned) cudaFree(q);
    delete p;
}
template <class FT> void* poisson_storage(PoissonPlan<FT>* p) { return p->kind == 2 ? (void*)p->source : (void*)p->storage; }
template <class FT> int poisson_kind(PoissonPlan<FT>* p) { return p->kind; }

template <class FT> static void launch_lines(FftArgs<FT>& A, int mode, bool contiguous_lines);

template <class FT>
static void run_pass(PoissonPlan<FT>* p, typename Cx<FT>::T* data, int d, int mode, const GridD<FT>* gphi, FT* phi_p0) {
    using CT = typename Cx<FT>::T;
    FftArgs<FT> A;
    int Nx = p->N[0], Ny = p->N[1], Nz = p->N[2];
    long long st[3] = {1, Nx, (long long)Nx * Ny};
    A.data = data; A.n = p->N[d]; A.log2n = p->log2n[d]; A.stride = st[d];
    A.dimL = d;
    if (d == 0) { A.dimA = 1; A.dimB = 2; } else if (d == 1) { A.dimA = 0; A.dimB = 2; } else { A.dimA = 0; A.dimB = 1; }
    A.nA = p->N[A.dimA]; A.nB = p->N[A.dimB];
    A.strideA = st[A.dimA]; A.strideB = st[A.dimB];
    A.kind = p->tkind[d]; A.tw = p->tw[d];
    A.M = p->M[d]; A.log2M = p->log2M[d]; A.bhat = p->bhat[d];
    const bool is_dct = A.kind == TK_DCT || A.kind == TK_DCT_POW2 || A.kind == TK_DCT_BLUE;
    A.scale = is_dct ? (FT)(1.0 / (2.0 * A.n)) : (FT)(1.0 / A.n);
    for (int q = 0; q < 3; ++q) A.lam[q] = p->lam[q];
    A.phi_p0 = phi_p0;
    if (gphi) for (int q = 0; q < 3; ++q) A.phi_st[q] = gphi->st[q];
    launch_lines<FT>(A, mode, d == 0);
}

// lines per block and launch of fft_lines_kernel for a filled argument block
template <class FT>
static void launch_lines(FftArgs<FT>& A, int mode, bool contiguous_lines) {
    using CT = typename Cx<FT>::T;
    const bool blue = A.kind == TK_BLUE || A.kind == TK_DCT_BLUE, direct = A.kind == TK_DFT || A.kind == TK_DCT;
    A.pad = 1;
    int LS = (blue ? A.M : A.n) + A.pad;
    int nbuf = direct ? 2 : 1;
    int ntw = A.kind == TK_POW2 ? A.n / 2 : A.kind == TK_DFT ? A.n : A.kind == TK_DCT ? 4 * A.n
            : A.kind == TK_DCT_POW2 ? A.n / 2 + A.n : A.kind == TK_BLUE ? A.M / 2 + A.n : A.M / 2 + 2 * A.n;
    // lines per block: 8 adjacent lines = 128-byte runs of the strided passes; more lines per block mean fewer resident
    // blocks to cover the per-stage barriers (256^3, ms per solve: T = 16 2.83, 8 2.32, 4 2.37; 512 threads 2.39)
    int T = 8;
    while (T > 1 && ((size_t)nbuf * T * LS + ntw) * sizeof(CT) > 96 * 1024) T >>= 1;
    if (contiguous_lines) { int Tm = std::max(1, 4096 / A.n); T = std::min(T, Tm); }
    T = std::min(T, A.nA);
    A.T = T;
    size_t smem = ((size_t)nbuf * T * LS + ntw) * sizeof(CT);
    dim3 grd(cdiv(A.nA, T), A.nB);
    auto launch = [&](auto kern) {
        OB_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
        kern<<<grd, 256, smem, stream()>>>(A);
        OB_LAUNCH_CHECK();
    };
    if (smem > 200 * 1024) throw Error("transform line too long for shared memory");
    if (mode == MODE_FWD) launch(fft_lines_kernel<FT, MODE_FWD>);
    else if (mode == MODE_INV) launch(fft_lines_kernel<FT, MODE_INV>);
    else launch(fft_lines_kernel<FT, MODE_FWD_DIV_INV>);
}

template <class FT>
void poisson_solve(PoissonPlan<FT>* p, const GridD<FT>& g, FT* phi_p0) {
    using CT = typename Cx<FT>::T;
    // plans that own only the half-spectrum fast path (and slab-decomposed plans) have no complex general storage:
    // they are driven through poisson_solve_velocities / poisson_solve_real
    if (poisson_storage<FT>(p) == nullptr)
        throw Error("this Poisson plan has no general complex storage: pass a right-hand side (ob200_poisson_solve with rhs != NULL) "
                    "or use ob200_solve_for_pressure");
    int dims[3], nd = 0;
    for (int d = 0; d < 3; ++d)
        if (p->topo[d] != OB_FLAT && !(p->kind == 2 && d == 2)) dims[nd++] = d;
    if (p->kind == 1) {
        if (nd == 0) throw Error("FFTBasedPoissonSolver needs at least one non-Flat dimension");
        for (int q = 0; q < nd - 1; ++q) run_pass(p, p->storage, dims[q], MODE_FWD, (const GridD<FT>*)nullptr, (FT*)nullptr);
        if (nd == 1) {
            run_pass(p, p->storage, dims[0], MODE_FWD_DIV_INV, &g, phi_p0);
        } else {
            run_pass(p, p->storage, dims[nd - 1], MODE_FWD_DIV_INV, (const GridD<FT>*)nullptr, (FT*)nullptr);
            for (int q = nd - 2; q >= 1; --q) run_pass(p, p->storage, dims[q], MODE_INV, (const GridD<FT>*)nullptr, (FT*)nullptr);
            run_pass(p, p->storage, dims[0], MODE_INV, &g, phi_p0);
        }
        return;
    }
    // Fourier-tridiagonal: forward xy on the source term, Thomas in z, backward xy, real, minus mean
    int Nx = p->N[0], Ny = p->N[1], Nz = p->N[2];
    for (int q = 0; q < nd; ++q) run_pass(p, p->source, dims[q], MODE_FWD, (const GridD<FT>*)nullptr, (FT*)nullptr);
    {
        dim3 blk(64), grd(cdiv(Nx, 64), Ny);
        thomas_kernel<FT, CT, true><<<grd, blk, 0, stream()>>>(Nx, Ny, Nz, p->lower, nullptr, p->lower,
                                                                p->lam[0], p->lam[1], p->dzF, p->dzC,
                                                                p->source, p->storage, p->scratch);
        OB_LAUNCH_CHECK();
    }
    for (int q = nd - 1; q >= 0; --q) run_pass(p, p->storage, dims[q], MODE_INV, (const GridD<FT>*)nullptr, (FT*)nullptr);
    long long tot = (long long)Nx * Ny * Nz;
    int blocks = (int)std::min<long long>(MEAN_BLOCKS, (tot + 255) / 256);
    sum_real_kernel<FT><<<blocks, 256, 0, stream()>>>(p->storage, tot, p->msum);
    OB_LAUNCH_CHECK();
    sub_mean_copy_kernel<FT><<<blocks, 256, 0, stream()>>>(p->storage, Nx, Ny, Nz, p->msum, blocks, phi_p0, g.st[0], g.st[1], g.st[2]);
    OB_LAUNCH_CHECK();
}

template <class FT> bool poisson_has_fast(PoissonPlan<FT>* p) { return p->fast != nullptr; }
template <class FT>
void poisson_solve_velocities(PoissonPlan<FT>* p, const GridD<FT>& g, const FT* u, const FT* v, const FT* w,
                              FT dt, FT* phi_p0) {
    ff::fast_poisson_solve<FT>(p->fast, g, u, v, w, dt, nullptr, phi_p0);
}
template <class FT>
void poisson_solve_real(PoissonPlan<FT>* p, const GridD<FT>& g, const FT* rhs, FT* phi_p0) {
    ff::fast_poisson_solve<FT>(p->fast, g, nullptr, nullptr, nullptr, FT(1), rhs, phi_p0);
}

#define INST(FT)                                                                                           \
    template bool poisson_has_fast<FT>(PoissonPlan<FT>*);                                                  \
    template void poisson_solve_velocities<FT>(PoissonPlan<FT>*, const GridD<FT>&, const FT*, const FT*,   \
                                               const FT*, FT, FT*);                                        \
    template void poisson_solve_real<FT>(PoissonPlan<FT>*, const GridD<FT>&, const FT*, FT*);              \
    template PoissonPlan<FT>* poisson_plan_create<FT>(const GridD<FT>&, int, const double*, const double*); \
    template void poisson_plan_destroy<FT>(PoissonPlan<FT>*);                                              \
    template void* poisson_storage<FT>(PoissonPlan<FT>*);                                                  \
    template int poisson_kind<FT>(PoissonPlan<FT>*);                                                       \
    template void poisson_solve<FT>(PoissonPlan<FT>*, const GridD<FT>&, FT*);
INST(float)
INST(double)

}  // namespace ob
