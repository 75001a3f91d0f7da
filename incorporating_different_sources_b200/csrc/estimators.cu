// Sibling estimators that reuse the batched Gram + batched Cholesky machinery (SURVEY 8(f) rank 3).
//
// lw_shrink_kernel: Ledoit-Wolf shrinkage of the sample covariance, the covariance estimator of
//   calculate_shrinkage_portfolio (portfolio_calculations.py:703-758): pypfopt 1.5.5
//   risk_models.CovarianceShrinkage(X, returns_data=True).ledoit_wolf() (:727-729) hands the excess returns to
//   sklearn.covariance.ledoit_wolf, whose published algorithm is restated here:
//       X_c = X - mean,  emp = X_c'X_c / m,  mu = tr(emp)/N,
//       delta_ = ||X_c'X_c||_F^2 / m^2,   beta_ = sum_k (sum_i X_c[k,i]^2)^2   (= sum of all entries of (X_c^2)'(X_c^2)),
//       beta = (beta_/m - delta_) / (N m),  delta = (delta_ - 2 mu tr(emp) + N mu^2) / N,
//       shrinkage = min(beta, delta) / delta,   Sigma = (1 - shrinkage) emp + shrinkage mu I.
//   The reference's closed form (its own CHECK, :748-756) is weights = (1/gamma) Sigma^-1 mu_hat; the annualisation
//   factor multiplies Sigma and mu_hat alike and cancels.  With C = X_c'X_c (left in the solver workspace by the Gram
//   stage) m Sigma = (1 - shrinkage) C + shrinkage mu m I, and (m Sigma) w = t = m mu_hat is solved by the unchanged
//   Cholesky kernel as (C + rho I) w = t / (1 - shrinkage), rho = shrinkage mu m / (1 - shrinkage): only the diagonal of
//   the workspace and the right-hand side are rewritten (a full rescaling pass would re-read and re-write 2 MB per window).
//   Two cases follow sklearn where that form does not apply: one asset (N = 1) has shrinkage 0, and a clipped window
//   (beta >= delta, shrinkage exactly 1) has Sigma = mu I, solved as mu m I w = t: its lower triangle is rewritten to
//   zero off the diagonal and mu m on it, and rhs = t.
//   The only O(m N) work is beta_: one pass over the window's rows (L2 resident: consecutive windows share them).
#include "common.cuh"
#include "kernels.h"

namespace bp {

constexpr int LW_THREADS = 256;
constexpr int LW_WARPS = LW_THREADS / 32;

__global__ void __launch_bounds__(LW_THREADS) lw_shrink_kernel(ShrinkParams p) {
    extern __shared__ __align__(16) double lw_sm[];
    double* xbar = lw_sm;                  // [ldv]
    double* scratch = xbar + p.ldv;        // [40]
    __shared__ double sh_scale, sh_diag;
    __shared__ bool sh_clip;

    const int w = blockIdx.x, tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int N = p.n_assets, K = p.n_window - 1;
    const double m = (double)K;
    const int day_row = p.day_row[w];
    const int extra_row = p.extra_row ? p.extra_row[w] : -1;
    const int K1 = extra_row >= 0 ? K - 1 : K;
    const long long r0 = (long long)day_row - K1 + 1;
    const double expo = ((double)p.span_days[w] / m) / 365.0;      // gbar / 365  (:40-48)
    for (int j = tid; j < p.ldv; j += LW_THREADS) xbar[j] = j < N ? p.t[(long long)w * p.ldv + j] / m : 0.0;
    __syncthreads();

    // ---- beta_ = sum_k ||x_k - xbar||^4: one warp per PAIR of rows (two independent load streams), 16-byte global
    // and shared loads, 4 column chunks in flight per row
    double b4 = 0.0;
    for (int k = 2 * warp; k < K; k += 2 * LW_WARPS) {
        const bool two = k + 1 < K;
        const long long ra = k < K1 ? r0 + k : (long long)extra_row;
        const long long rb = !two ? ra : (k + 1 < K1 ? r0 + k + 1 : (long long)extra_row);
        const double aa = pow(1.0 + p.rf_row[ra], expo) - 1.0;
        const double ab = pow(1.0 + p.rf_row[rb], expo) - 1.0;
        const double* rowa = p.lr_daily + ra * p.ld;
        const double* rowb = p.lr_daily + rb * p.ld;
        double sa = 0.0, sb = 0.0;
#pragma unroll 4
        for (int c = 2 * lane; c < p.ldv; c += 64) {      // pad columns: returns and xbar are zero, d = -a is masked
            const double2 va = *reinterpret_cast<const double2*>(rowa + c);
            const double2 vb = *reinterpret_cast<const double2*>(rowb + c);
            const double2 xb = *reinterpret_cast<const double2*>(xbar + c);
            const double m0 = c < N ? 1.0 : 0.0, m1 = c + 1 < N ? 1.0 : 0.0;
            const double a0 = m0 * ((va.x - aa) - xb.x), a1 = m1 * ((va.y - aa) - xb.y);
            const double b0 = m0 * ((vb.x - ab) - xb.x), b1 = m1 * ((vb.y - ab) - xb.y);
            sa = fma(a0, a0, sa);
            sa = fma(a1, a1, sa);
            sb = fma(b0, b0, sb);
            sb = fma(b1, b1, sb);
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            sa += __shfl_xor_sync(0xffffffffu, sa, o);
            sb += __shfl_xor_sync(0xffffffffu, sb, o);
        }
        if (lane == 0) {
            b4 = fma(sa, sa, b4);
            if (two) b4 = fma(sb, sb, b4);
        }
    }
    const double beta_ = block_sum(b4, scratch);

    // ---- trace and squared Frobenius norm of C from its lower triangle
    double* S = p.S + (long long)w * p.win_stride;
    double tr = 0.0, fr = 0.0;
    for (int i = warp; i < N; i += LW_WARPS) {
        const double* row = S + (long long)i * p.ldS;
        for (int j = lane; j <= i; j += 32) {
            const double v = row[j];
            if (j == i) {
                tr += v;
                fr = fma(v, v, fr);
            } else {
                fr = fma(2.0 * v, v, fr);
            }
        }
    }
    tr = block_sum(tr, scratch);
    fr = block_sum(fr, scratch);

    if (tid == 0) {
        const double Nd = (double)N;
        const double trace_e = tr / m;
        const double mu = trace_e / Nd;
        const double delta_ = fr / (m * m);
        double beta = 1.0 / (Nd * m) * (beta_ / m - delta_);
        double delta = delta_ - 2.0 * mu * trace_e + Nd * mu * mu;
        delta /= Nd;
        const double beta_raw = beta;
        beta = fmin(beta, delta);
        // sklearn: shrinkage 0 for one feature (delta is 0 in exact arithmetic there, rounding leaves it either sign)
        const double shrink = (N == 1 || beta == 0.0) ? 0.0 : beta / delta;
        double* scal = p.scal + (long long)w * BP_S_COUNT;
        scal[BP_S_LW_SHRINKAGE] = shrink;
        scal[BP_S_LW_MU] = mu;
        scal[BP_S_LW_BETA] = beta_raw;
        scal[BP_S_LW_DELTA] = delta;
        // beta >= delta (also any delta <= 0 left by rounding) clips the intensity to exactly 1: Sigma_LW = mu I, and
        // the window's system is m Sigma_LW w = mu m I w = t (1/(1 - shrink) would be inf)
        sh_clip = shrink == 1.0;
        sh_scale = sh_clip ? 1.0 : 1.0 / (1.0 - shrink);
        sh_diag = sh_clip ? mu * m : shrink * mu * m / (1.0 - shrink);
    }
    __syncthreads();
    const double scale = sh_scale, diag = sh_diag;
    if (sh_clip) {                                       // uniform per block; only clipped windows pay the O(N^2) write
        for (int i = warp; i < N; i += LW_WARPS) {
            double* row = S + (long long)i * p.ldS;
            for (int j = lane; j <= i; j += 32) row[j] = j == i ? diag : 0.0;
        }
    } else {
        for (int i = tid; i < N; i += LW_THREADS) S[(long long)i * p.ldS + i] += diag;
    }
    for (int j = tid; j < p.ldv; j += LW_THREADS) p.rhs[(long long)w * p.ldv + j] = j < N ? scale * p.t[(long long)w * p.ldv + j] : 0.0;
}

cudaError_t launch_lw_shrink(const ShrinkParams& p, cudaStream_t st) {
    if (p.n_windows <= 0) return cudaSuccess;
    const size_t smem = sizeof(double) * (size_t)(p.ldv + 40);
    lw_shrink_kernel<<<p.n_windows, LW_THREADS, smem, st>>>(p);
    return cudaGetLastError();
}

}  // namespace bp
