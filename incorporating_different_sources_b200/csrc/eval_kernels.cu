// Evaluation statistics of a path ensemble (portfolio_evaluation.py:464-701, performance_metrics): for every return
// series of an ensemble (64 synthetic paths x strategies, BASELINE config 5) the scalars the reference computes one
// pandas / QuantStats call at a time -- cumulative return, CAGR, Sharpe, Sortino, Calmar, maximum drawdown, average
// win / loss / return, best / worst day, annualised volatility, parametric daily VaR, and the skewness / kurtosis /
// per-period Sharpe ratio that its probabilistic Sharpe ratio (:78-120) is built from.
//
// One CTA per series; reductions in a fixed order (bit-reproducible), the drawdown through a chunked scan of the
// cumulative product (each thread owns a contiguous chunk; the chunk products and chunk maxima are combined by one
// thread in index order).  HBM bound and tiny: T = 4,149 returns per series; the point is that a path ensemble never
// goes back to pandas.  Formulas: QuantStats 0.0.62 (requirements.txt:10, not vendored) as restated in
// oracle/eval_oracle.py, which pins them on the reference's own CHECK expressions (:520-650).
#include <cfloat>

#include "common.cuh"
#include "../../include/bayes_portfolio.h"
#include "kernels.h"

namespace bp {

constexpr int PM_THREADS = 256;

__device__ __forceinline__ double block_max(double v, double* s8) {
    for (int o = 16; o > 0; o >>= 1) v = fmax(v, __shfl_xor_sync(0xffffffffu, v, o));
    __syncthreads();
    if ((threadIdx.x & 31) == 0) s8[threadIdx.x >> 5] = v;
    __syncthreads();
    double r = s8[0];
    for (int k = 1; k < PM_THREADS / 32; ++k) r = fmax(r, s8[k]);
    return r;
}

__global__ void __launch_bounds__(PM_THREADS) path_metrics_kernel(PathMetricsParams p) {
    __shared__ double scratch[40];
    __shared__ double s8[PM_THREADS / 32];
    __shared__ double cprod[PM_THREADS], cmax[PM_THREADS], cbase[PM_THREADS], cpeak[PM_THREADS];
    const int tid = threadIdx.x;
    const int T = p.n_obs;
    const double* r = p.returns + (long long)blockIdx.x * p.ld;
    const double* x = p.excess + (long long)blockIdx.x * p.ld;
    double* out = p.out + (long long)blockIdx.x * BP_PM_COUNT;

    // ---- pass 1: sums, extremes, conditional sums
    double sr = 0, sx = 0, sneg = 0, cneg = 0, spos = 0, cpos = 0, snz = 0, cnz = 0, dn2 = 0, mx = -INFINITY, mn = INFINITY;
    for (int i = tid; i < T; i += PM_THREADS) {
        const double ri = r[i], xi = x[i];
        sr += ri;
        sx += xi;
        if (ri < 0) { sneg += ri; cneg += 1; }
        if (ri > 0) { spos += ri; cpos += 1; }
        if (ri != 0) { snz += ri; cnz += 1; }
        if (xi < 0) dn2 = fma(xi, xi, dn2);
        mx = fmax(mx, ri);
        mn = fmin(mn, ri);
    }
    sr = block_sum(sr, scratch);   sx = block_sum(sx, scratch);
    sneg = block_sum(sneg, scratch); cneg = block_sum(cneg, scratch);
    spos = block_sum(spos, scratch); cpos = block_sum(cpos, scratch);
    snz = block_sum(snz, scratch);  cnz = block_sum(cnz, scratch);
    dn2 = block_sum(dn2, scratch);
    mx = block_max(mx, s8);
    mn = -block_max(-mn, s8);
    const double n = (double)T, mr = sr / n, mxs = sx / n;

    // ---- pass 2: central moments (x1 = sum of the excess deviations, for the flat-sample rule of the skewness)
    double r2 = 0, x1 = 0, x2 = 0, x3 = 0, x4 = 0;
    for (int i = tid; i < T; i += PM_THREADS) {
        const double a = r[i] - mr, b = x[i] - mxs, b2 = b * b;
        r2 = fma(a, a, r2);
        x1 += b;
        x2 += b2;
        x3 = fma(b2, b, x3);
        x4 = fma(b2, b2, x4);
    }
    r2 = block_sum(r2, scratch); x2 = block_sum(x2, scratch); x3 = block_sum(x3, scratch); x4 = block_sum(x4, scratch);
    x1 = block_sum(x1, scratch);

    // ---- cumulative product and drawdown: contiguous chunk per thread
    const int chunk = (T + PM_THREADS - 1) / PM_THREADS;
    const int i0 = min(tid * chunk, T), i1 = min(i0 + chunk, T);
    double prod = 1.0, lmax = -INFINITY;
    for (int i = i0; i < i1; ++i) {
        prod *= 1.0 + r[i];
        lmax = fmax(lmax, prod);
    }
    cprod[tid] = prod;
    cmax[tid] = lmax;
    __syncthreads();
    if (tid == 0) {
        double base = 1.0, peak = -INFINITY;
        for (int t = 0; t < PM_THREADS; ++t) {
            cbase[t] = base;                          // product of everything before chunk t
            cpeak[t] = peak;                          // running maximum before chunk t
            peak = fmax(peak, base * cmax[t]);
            base *= cprod[t];
        }
        cprod[0] = base;                              // total product
    }
    __syncthreads();
    const double total = cprod[0];
    double cum = cbase[tid], peak = cpeak[tid], dd = INFINITY;
    for (int i = i0; i < i1; ++i) {
        cum *= 1.0 + r[i];
        peak = fmax(peak, cum);
        dd = fmin(dd, cum / peak);
    }
    const double mdd = -block_max(-dd, s8) - 1.0;

    if (tid == 0) {
        const double sd_r = sqrt(r2 / (n - 1.0)), sd_x = sqrt(x2 / (n - 1.0));
        const double cagr = pow(fabs(total), 1.0 / p.years) - 1.0;
        const double nan = __longlong_as_double(0x7ff8000000000000LL);
        out[BP_PM_CUM_RETURN] = total - 1.0;
        out[BP_PM_CAGR] = cagr;
        out[BP_PM_SHARPE] = mxs / sd_x * sqrt(252.0);
        out[BP_PM_SORTINO] = mxs / sqrt(dn2 / n) * sqrt(252.0);
        out[BP_PM_MAX_DD] = mdd;
        out[BP_PM_CALMAR] = cagr / fabs(mdd);
        out[BP_PM_AVG_LOSS] = cneg > 0 ? sneg / cneg : nan;
        out[BP_PM_AVG_RETURN] = cnz > 0 ? snz / cnz : nan;
        out[BP_PM_AVG_WIN] = cpos > 0 ? spos / cpos : nan;
        out[BP_PM_BEST] = mx;
        out[BP_PM_WORST] = mn;
        out[BP_PM_ANN_VOL] = sd_r * sqrt(252.0);
        out[BP_PM_DAILY_VAR] = fma(sd_r, -1.6448536269514729, mr);     // norm.ppf(0.05, mu, sigma)
        const double m2 = x2 / n;
        // scipy's rule: NaN when m2 <= (eps mean)^2.  It is tested on the two-pass corrected m2, from which the
        // error of the mean cancels: a constant series whose computed mean is a few ulp off has b = delta != 0 in
        // every term, so x2 / n = delta^2 would pass for a spread (and give skew = +-1, kurtosis = 1).
        const double m2c = (x2 - x1 * x1 / n) / n, eps_mean = DBL_EPSILON * mxs;
        const bool flat = m2c <= eps_mean * eps_mean;
        out[BP_PM_SKEW] = flat ? nan : (x3 / n) / (m2 * sqrt(m2));      // scipy.stats.skew (biased)
        out[BP_PM_KURT] = flat ? nan : (x4 / n) / (m2 * m2);            // scipy.stats.kurtosis(fisher=False)
        out[BP_PM_SHARPE_1] = mxs / sd_x;                               // periods = 1 (:81-82)
    }
}

cudaError_t launch_path_metrics(const PathMetricsParams& p, cudaStream_t st) {
    if (p.n_paths <= 0) return cudaSuccess;
    path_metrics_kernel<<<p.n_paths, PM_THREADS, 0, st>>>(p);
    return cudaGetLastError();
}

}  // namespace bp
