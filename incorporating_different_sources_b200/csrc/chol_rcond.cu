// Reciprocal condition number of every factorised window: LAPACK's dpocon on the Cholesky factor the solver leaves in
// the workspace.  A positive pivot only says the factorisation finished; a window with cond_1 = 1e13 passes it and
// returns weights with hardly a correct digit.  dpocon estimates ||A^-1||_1 from a few solves with the factor
// (dlacn2, Hager-Higham), so the estimate costs a few passes over L instead of an inverse.
//
//   sym_norm1_kernel   anorm1 = max_j sum_i |A_ij| of the symmetric A of the lower triangle, BEFORE the factorisation
//                      overwrites it: one CTA per window, one read of the triangle, fixed summation order (lower part
//                      of column j top-down by the lane of j, upper part as row j of the triangle by one warp sum).
//   chol_rcond_kernel  dlacn2's state machine (ITMAX = 5, x >= 0 -> +1, first-index idamax) with A^-1 v = L'^-1 L^-1 v,
//                      one CTA per window, v in shared memory, forward and back substitution in the 32-block form of
//                      chol_panel.cuh.  dlacn2's final vector (alternating signs, 1 + i/(N-1)) does not depend on the
//                      iteration, so it rides along with the first vector (one pass over L for both): every window
//                      takes one pass fewer than dpocon's sequence of solves, with the same result.
//   rcond = (1 / est) / anorm1; 0 when the status is non-zero (incomplete factor), anorm1 is not positive, or a solve
//   gives a non-finite 1-norm (dpocon's overflow exit).
#include <algorithm>
#include <cstdlib>

#include "chol_panel.cuh"

namespace bp {

using namespace chol;

namespace {

constexpr int NORM_WARPS = 8;
constexpr int NORM_THREADS = NORM_WARPS * 32;
constexpr int RC_WARPS = 4;
constexpr int RC_THREADS = RC_WARPS * 32;
constexpr int RC_ITMAX = 5;

__device__ __forceinline__ int round_nb(int n) { return (n + NB - 1) / NB * NB; }

}  // namespace

__global__ void __launch_bounds__(NORM_THREADS) sym_norm1_kernel(const SolveParams p) {
    extern __shared__ double colsum[];      // [Nr]
    __shared__ double scratch[40];
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int N = p.n_assets, ld = p.ldS;
    const int w = blockIdx.x * max(p.w_stride, 1);
    const double* S = p.S + (long long)w * p.win_stride;
    // lower part, rows i >= j: warp k owns the columns 32 (k + NORM_WARPS c) + lane, coalesced rows
    for (int b = warp; b * NB < N; b += NORM_WARPS) {
        const int j = NB * b + lane;
        double s = 0.0;
        for (int i = NB * b; i < N; ++i)
            if (j <= i) s += fabs(S[(long long)i * ld + j]);
        colsum[j] = s;
    }
    __syncthreads();
    // upper part of column i = row i of the triangle left of the diagonal, one warp per row
    for (int i = warp; i < N; i += NORM_WARPS) {
        double s = 0.0;
        for (int j = lane; j < i; j += 32) s += fabs(S[(long long)i * ld + j]);
        s = warp_sum(s);
        if (lane == 0) colsum[i] += s;
    }
    __syncthreads();
    double m = 0.0;
    for (int j = tid; j < N; j += NORM_THREADS) {
        const double v = colsum[j];
        if (v > m || v != v) m = v;        // a NaN entry makes the norm NaN
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        const double v = __shfl_xor_sync(0xffffffffu, m, o);
        if (v > m || v != v) m = v;
    }
    if (lane == 0) scratch[warp] = m;
    __syncthreads();
    if (tid == 0) {
        for (int k = 1; k < NORM_WARPS; ++k)
            if (scratch[k] > m || scratch[k] != scratch[k]) m = scratch[k];
        p.scal[(long long)w * BP_S_COUNT + BP_S_ANORM1] = m;
    }
}

namespace {

// x[r] <- A^-1 x[r] = L'^-1 L^-1 x[r] for r < NRHS, in place in x[NRHS][Nr] (zero beyond N)
template <int NRHS>
__device__ void llt_solve(double* x, double* P, const double* S, int ld, int N, int Nr, int warp, int lane) {
    const int nb = Nr / NB;
    __syncthreads();                        // x is complete
    for (int b = 0; b < nb; ++b) {
        load_diag_block<RC_WARPS>(P, S, ld, b, N, warp, lane);
        forward_reduce_block<NRHS, RC_WARPS>(x, x, S, ld, Nr, N, b, warp, lane);
        __syncthreads();
        if (warp < NRHS) {
            double* v = x + warp * Nr + NB * b + lane;
            *v = solve_diag_block_lower(*v, P, lane);
        }
        __syncthreads();
    }
    for (int b = nb - 1; b >= 0; --b) {
        load_diag_block<RC_WARPS>(P, S, ld, b, N, warp, lane);
        __syncthreads();
        if (warp < NRHS) {
            double* v = x + warp * Nr + NB * b + lane;
            *v = solve_diag_block(*v, P, lane);
        }
        __syncthreads();
        for (int bb = warp; bb < b; bb += RC_WARPS) reduce_block<NRHS>(x, x, S, ld, Nr, N, b, NB * bb + lane);
    }
    __syncthreads();
}

__device__ double block_asum(const double* x, int N, double* scratch) {
    double s = 0.0;
    for (int j = threadIdx.x; j < N; j += RC_THREADS) s += fabs(x[j]);
    return block_sum(s, scratch);
}

// first index of the largest |x_j| (BLAS idamax), for every thread
__device__ int block_idamax(const double* x, int N, double* sv, int* si) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    double bv = -1.0;
    int bi = 0;
    for (int j = threadIdx.x; j < N; j += RC_THREADS) {
        const double a = fabs(x[j]);
        if (a > bv) {
            bv = a;
            bi = j;
        }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        const double ov = __shfl_xor_sync(0xffffffffu, bv, o);
        const int oi = __shfl_xor_sync(0xffffffffu, bi, o);
        if (ov > bv || (ov == bv && oi < bi)) {
            bv = ov;
            bi = oi;
        }
    }
    __syncthreads();
    if (lane == 0) {
        sv[warp] = bv;
        si[warp] = bi;
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        for (int k = 1; k < RC_WARPS; ++k)
            if (sv[k] > bv || (sv[k] == bv && si[k] < bi)) {
                bv = sv[k];
                bi = si[k];
            }
        si[RC_WARPS] = bi;
    }
    __syncthreads();
    return si[RC_WARPS];
}

// x <- sign(x) (x >= 0 -> +1, dlacn2), and the same in isgn
__device__ void take_signs(double* x, signed char* isgn, int N) {
    for (int j = threadIdx.x; j < N; j += RC_THREADS) {
        const bool pos = x[j] >= 0.0;
        x[j] = pos ? 1.0 : -1.0;
        isgn[j] = pos ? 1 : -1;
    }
}

// 1 when sign(x) equals isgn everywhere, for every thread
__device__ bool same_signs(const double* x, const signed char* isgn, int N) {
    bool same = true;
    for (int j = threadIdx.x; j < N; j += RC_THREADS) same = same && (x[j] >= 0.0 ? 1 : -1) == isgn[j];
    return __syncthreads_and(same) != 0;
}

// dlacn2's estimate of ||A^-1||_1 for one window (every thread returns it); 0 after a non-finite solve
__device__ double inv_norm1_estimate(double* x, signed char* isgn, double* P, const double* S, int ld, int N, int Nr,
                                     double* scratch, int* iscratch, int warp, int lane) {
    const double invn = 1.0 / (double)N;
    for (int j = threadIdx.x; j < Nr; j += RC_THREADS) {
        const double alt = N > 1 ? (j & 1 ? -1.0 : 1.0) * (1.0 + (double)j / (double)(N - 1)) : 1.0;
        x[j] = j < N ? invn : 0.0;
        x[Nr + j] = j < N ? alt : 0.0;
    }
    llt_solve<2>(x, P, S, ld, N, Nr, warp, lane);
    double est = block_asum(x, N, scratch);
    const double alt_norm = block_asum(x + Nr, N, scratch);
    if (!isfinite(est) || !isfinite(alt_norm)) return 0.0;
    if (N == 1) return est;
    const double alt_est = 2.0 * (alt_norm / (double)(3 * N));

    take_signs(x, isgn, N);
    llt_solve<1>(x, P, S, ld, N, Nr, warp, lane);
    if (!isfinite(block_asum(x, N, scratch))) return 0.0;
    int j = block_idamax(x, N, scratch, iscratch);
    for (int iter = 2;; ++iter) {
        for (int k = threadIdx.x; k < Nr; k += RC_THREADS) x[k] = k == j ? 1.0 : 0.0;
        llt_solve<1>(x, P, S, ld, N, Nr, warp, lane);
        const double estold = est;
        est = block_asum(x, N, scratch);
        if (!isfinite(est)) return 0.0;
        if (same_signs(x, isgn, N) || est <= estold) break;      // repeated sign vector, or cycling
        take_signs(x, isgn, N);
        llt_solve<1>(x, P, S, ld, N, Nr, warp, lane);
        if (!isfinite(block_asum(x, N, scratch))) return 0.0;
        const int jlast = j;
        j = block_idamax(x, N, scratch, iscratch);
        const bool more = x[jlast] != fabs(x[j]) && iter < RC_ITMAX;
        __syncthreads();                    // x is rewritten next
        if (!more) break;
    }
    return alt_est > est ? alt_est : est;
}

}  // namespace

__global__ void __launch_bounds__(RC_THREADS) chol_rcond_kernel(const SolveParams p) {
    extern __shared__ double sm[];
    __shared__ double scratch[40];
    __shared__ int iscratch[RC_WARPS + 1];
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int N = p.n_assets, ld = p.ldS, Nr = round_nb(N);
    double* P = sm;                         // [NB][LDQ] diagonal block
    double* x = P + NB * LDQ;               // [2][Nr]
    signed char* isgn = reinterpret_cast<signed char*>(x + 2 * Nr);   // [Nr]
    const int stride = max(p.w_stride, 1);
    for (int q = blockIdx.x; q < p.n_windows; q += gridDim.x) {
        const int w = q * stride;
        double* scal = p.scal + (long long)w * BP_S_COUNT;
        const double anorm = scal[BP_S_ANORM1];
        double rcond = 0.0;
        if (p.status[w] == 0 && anorm > 0.0) {
            const double est = inv_norm1_estimate(x, isgn, P, p.S + (long long)w * p.win_stride, ld, N, Nr, scratch,
                                                  iscratch, warp, lane);
            if (est != 0.0) rcond = (1.0 / est) / anorm;
        }
        if (tid == 0) scal[BP_S_RCOND] = rcond;
        __syncthreads();                    // shared memory is reused by the next window
    }
}

static size_t rcond_smem_bytes(int n_assets) {
    const size_t Nr = (size_t)(n_assets + NB - 1) / NB * NB;
    return sizeof(double) * (NB * LDQ + 2 * Nr) + Nr;
}

cudaError_t launch_sym_norm1(const SolveParams& p, cudaStream_t st) {
    if (p.n_windows <= 0) return cudaSuccess;
    const size_t smem = sizeof(double) * (size_t)((p.n_assets + NB - 1) / NB * NB);
    sym_norm1_kernel<<<p.n_windows, NORM_THREADS, smem, st>>>(p);
    return cudaGetLastError();
}

// CTAs of a launch: one per window, unless BP_RCOND_INFLIGHT_MB caps the factors in flight (CTAs x N^2 x 4 bytes) so
// that a window's factor can stay in L2 over its passes (the CTAs then loop over the windows)
static int rcond_grid(const SolveParams& p) {
    static const long long budget = [] {
        const char* e = getenv("BP_RCOND_INFLIGHT_MB");
        return e ? atoll(e) << 20 : 0LL;
    }();
    if (budget <= 0) return p.n_windows;
    const long long per = 4LL * p.n_assets * p.n_assets;
    const long long g = std::max(1LL, budget / per);
    return (int)std::min<long long>(g, p.n_windows);
}

cudaError_t launch_chol_rcond(const SolveParams& p, cudaStream_t st) {
    if (p.n_windows <= 0) return cudaSuccess;
    const size_t smem = rcond_smem_bytes(p.n_assets);
    cudaError_t e = cudaFuncSetAttribute(chol_rcond_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    chol_rcond_kernel<<<rcond_grid(p), RC_THREADS, smem, st>>>(p);
    return cudaGetLastError();
}

}  // namespace bp
