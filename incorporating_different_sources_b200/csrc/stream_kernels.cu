// Streaming (HBM / L2 bound) stages of the path.
//
//  * log_returns_kernel        : prices -> log(P_i / P_{i-1})           (portfolio_calculations.py:37, :314)
//  * hf_log_returns_kernel     : the same for the intraday rows, with the dropna of :314 (keep mask per row)
//  * window_prep_kernel        : per rebalance window, everything that is O(N*K):
//      a_k, t, u            (:40-57, :222)        excess-return column sums via the rank-2 form
//      n0, n1               (:90-114, :247-282)   MCM (VIX/EPU) scaling of the prior
//      w0                   (:361-380, :661-701)  value / equal prior weights
//      hbar, S0*w0, v0      (:314-318, :64-88)    HF realised-covariance mean terms, w0'S0w0
//      c, b = c*S0*w0 + t   (:415-418, :489)      conjugate scalar and right-hand side
//  * pack / unpack helpers between the padded device layout and dense N x N outputs.
//
// The excess-return matrix X_w = L - a_w 1' differs per window (SURVEY F3), but the Gram matrix
// never needs X_w explicitly:  T = L'L - u 1' - 1 u' + (a'a) 11',  u = L'a,  t = L'1 - (sum a) 1.
// The window_prep kernel produces p = u - (a'a)/2 so that T_ij = (L'L)_ij - p_i - p_j, which the
// Gram kernel applies in its epilogue; the shared log-return matrix L is then TMA-loadable by
// every overlapping window.
#include "common.cuh"
#include "kernels.h"

namespace bp {

// ------------------------------------------------------------------------------------------------
// P is the DENSE host layout [rows][ld_in = n_assets]; out is padded to ld_out (multiple of 16, the
// TMA / vector-load layout), pad columns are written as zero.  One thread per pair of columns.
template <bool VEC>
__global__ void log_returns_kernel(const double* __restrict__ P, int ld_in, double* __restrict__ out, int ld_out,
                                   long long row_begin, long long rows, int n_assets) {
    const int half = ld_out >> 1;
    const int c = (blockIdx.x * blockDim.x + threadIdx.x) * 2;
    if (c >= ld_out) return;
    for (long long r = row_begin + blockIdx.y; r < rows; r += gridDim.y) {
        double2 o = make_double2(0.0, 0.0);
        if (r > 0 && c < n_assets) {
            const double* cur = P + r * ld_in + c;
            const double* prv = cur - ld_in;
            if (VEC && c + 1 < n_assets) {
                const double2 p = *reinterpret_cast<const double2*>(cur);
                const double2 q = *reinterpret_cast<const double2*>(prv);
                o.x = log(p.x / q.x);
                o.y = log(p.y / q.y);
            } else {
                o.x = log(cur[0] / prv[0]);
                if (c + 1 < n_assets) o.y = log(cur[1] / prv[1]);
            }
        }
        *reinterpret_cast<double2*>(out + r * ld_out + c) = o;
    }
    (void)half;
}

// rows [row_begin, rows) of the return matrix (row 0 is the zero row; row r needs price rows r-1 and r)
void launch_log_returns(const double* P, int ld_in, double* out, int ld_out, long long rows, int n_assets,
                        int sm_count, cudaStream_t st, long long row_begin) {
    if (rows <= row_begin) return;
    const int threads = 128;
    const int bx = (ld_out / 2 + threads - 1) / threads;
    long long by = rows - row_begin;
    const long long cap = (long long)sm_count * 32 / bx + 1;
    if (by > cap) by = cap;
    if (by > 65535) by = 65535;
    dim3 grid(bx, (unsigned)by);
    if ((ld_in & 1) == 0)
        log_returns_kernel<true><<<grid, threads, 0, st>>>(P, ld_in, out, ld_out, row_begin, rows, n_assets);
    else
        log_returns_kernel<false><<<grid, threads, 0, st>>>(P, ld_in, out, ld_out, row_begin, rows, n_assets);
}

// Intraday returns with the reference's dropna (:314): a return row with a NaN in ANY column -- a NaN bar in price
// row r-1 or r, or a 0/0 or inf/inf quotient -- is dropped.  A dropped row is written as zeros, which add nothing to any
// sum the later stages form, and keep[r] = 0; a kept row is exactly log_returns_kernel's row.  One warp per row: the
// keep decision is a warp vote, so no block barrier holds the other rows back.  Row 0 has no return (keep[0] = 0).
template <bool VEC>
__global__ void __launch_bounds__(256, 6) hf_log_returns_kernel(const double* __restrict__ P, int ld_in, double* __restrict__ out,
                                                                int ld_out, unsigned char* __restrict__ keep, long long row_begin, long long rows, int n_assets) {
    const int lane = threadIdx.x & 31;
    const long long warps = (long long)gridDim.x * (blockDim.x >> 5);
    for (long long r = row_begin + blockIdx.x * (long long)(blockDim.x >> 5) + (threadIdx.x >> 5); r < rows; r += warps) {
        double* o_row = out + r * ld_out;
        bool nan = r == 0;
#pragma unroll 4
        for (int c = lane * 2; c < ld_out; c += 64) {
            double2 o = make_double2(0.0, 0.0);
            if (r > 0 && c < n_assets) {
                const double* cur = P + r * ld_in + c;
                const double* prv = cur - ld_in;
                if (VEC && c + 1 < n_assets) {
                    const double2 p = *reinterpret_cast<const double2*>(cur);
                    const double2 q = *reinterpret_cast<const double2*>(prv);
                    o.x = log(p.x / q.x);
                    o.y = log(p.y / q.y);
                } else {
                    o.x = log(cur[0] / prv[0]);
                    if (c + 1 < n_assets) o.y = log(cur[1] / prv[1]);
                }
            }
            nan |= isnan(o.x) || isnan(o.y);
            *reinterpret_cast<double2*>(o_row + c) = o;
        }
        const bool drop = __any_sync(0xffffffffu, nan);
        if (drop)
            for (int c = lane * 2; c < ld_out; c += 64) *reinterpret_cast<double2*>(o_row + c) = make_double2(0.0, 0.0);
        if (lane == 0) keep[r] = drop ? 0 : 1;
    }
}

void launch_hf_log_returns(const double* P, int ld_in, double* out, int ld_out, unsigned char* keep, long long row_begin,
                           long long rows, int n_assets, int sm_count, cudaStream_t st) {
    if (rows <= row_begin) return;
    const int threads = 256, rows_per_block = threads / 32;
    long long blocks = (rows - row_begin + rows_per_block - 1) / rows_per_block;
    if (blocks > (long long)sm_count * 6) blocks = (long long)sm_count * 6;     // one wave at the launch bounds
    if ((ld_in & 1) == 0)
        hf_log_returns_kernel<true><<<(unsigned)blocks, threads, 0, st>>>(P, ld_in, out, ld_out, keep, row_begin, rows, n_assets);
    else
        hf_log_returns_kernel<false><<<(unsigned)blocks, threads, 0, st>>>(P, ld_in, out, ld_out, keep, row_begin, rows, n_assets);
}

// ------------------------------------------------------------------------------------------------
// Warp-per-row column accumulation over rows [r0, r0+nr) of a row-major matrix with leading
// dimension ld, restricted to the 512-column block starting at col0.  Lane l owns columns
// col0 + 64*ch + 2*l (+1), ch = 0..7, so every row is read with coalesced 16-byte loads.
//   sum[ch]  += x            wsum[ch] += wgt[k] * x            (wgt may be null)
//   if DOT:  y[k] (+)= sum_c x_c * w0[c]   (row dot with a shared-memory vector)
constexpr int PREP_THREADS = 256;
constexpr int PREP_WARPS = PREP_THREADS / 32;
constexpr int NCH = 8;

template <bool DOT>
__device__ __forceinline__ void col_accumulate(const double* __restrict__ M, int ld, long long r0, int nr,
                                               int col0, const double* wgt, const double* w0s, double* y,
                                               bool y_accumulate, double2 (&sum)[NCH], double2 (&wsum)[NCH]) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
    for (int ch = 0; ch < NCH; ++ch) {
        sum[ch] = make_double2(0.0, 0.0);
        wsum[ch] = make_double2(0.0, 0.0);
    }
    for (int k = warp; k < nr; k += PREP_WARPS) {
        const double* row = M + (r0 + k) * (long long)ld + col0;
        const double wk = wgt ? wgt[k] : 0.0;
        double dot = 0.0;
#pragma unroll
        for (int ch = 0; ch < NCH; ++ch) {
            const int c = ch * 64 + lane * 2;
            if (col0 + c < ld) {
                const double2 x = *reinterpret_cast<const double2*>(row + c);
                sum[ch].x += x.x;
                sum[ch].y += x.y;
                wsum[ch].x = fma(wk, x.x, wsum[ch].x);
                wsum[ch].y = fma(wk, x.y, wsum[ch].y);
                if (DOT) dot = fma(x.x, w0s[col0 + c], fma(x.y, w0s[col0 + c + 1], dot));
            }
        }
        if (DOT) {
            dot = warp_sum(dot);
            if (lane == 0) y[k] = y_accumulate ? y[k] + dot : dot;
        }
    }
}

// Intraday rows in ONE pass (ld <= 512): per row k the warp holds the whole row in registers, reduces the dot
// y_k = h_k . w0 with shuffles and accumulates both sum_k h_k and sum_k y_k h_k = H'y.  The centred product the
// prior needs is H'(y - ybar) = H'y - ybar * (H'1), so the second sweep over the rows (10 GB of DRAM traffic per
// batch: with ~450 windows in flight the rows do not stay in L2) is not needed.
__device__ __forceinline__ void hf_single_pass(const double* __restrict__ M, int ld, long long r0, int nr,
                                               const double* w0s, double* y, double2 (&sum)[NCH], double2 (&wsum)[NCH]) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
    for (int ch = 0; ch < NCH; ++ch) {
        sum[ch] = make_double2(0.0, 0.0);
        wsum[ch] = make_double2(0.0, 0.0);
    }
    for (int k = warp; k < nr; k += PREP_WARPS) {
        const double* row = M + (r0 + k) * (long long)ld;
        double2 x[NCH];
#pragma unroll
        for (int ch = 0; ch < NCH; ++ch) {
            const int c = ch * 64 + lane * 2;
            x[ch] = c < ld ? *reinterpret_cast<const double2*>(row + c) : make_double2(0.0, 0.0);
        }
        double dot = 0.0;
#pragma unroll
        for (int ch = 0; ch < NCH; ++ch) {
            const int c = ch * 64 + lane * 2;
            if (c < ld) dot = fma(x[ch].x, w0s[c], fma(x[ch].y, w0s[c + 1], dot));
        }
        dot = warp_sum(dot);
        if (lane == 0) y[k] = dot;
#pragma unroll
        for (int ch = 0; ch < NCH; ++ch) {
            sum[ch].x += x[ch].x;
            sum[ch].y += x[ch].y;
            wsum[ch].x = fma(dot, x[ch].x, wsum[ch].x);
            wsum[ch].y = fma(dot, x[ch].y, wsum[ch].y);
        }
    }
}

// Cross-warp reduction of the per-lane column partials through shared memory `red`
// ([PREP_WARPS][512] doubles); thread j of the block ends up owning columns col0+2j, col0+2j+1.
__device__ __forceinline__ double2 reduce_cols(const double2 (&part)[NCH], double* red) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    __syncthreads();
#pragma unroll
    for (int ch = 0; ch < NCH; ++ch)
        *reinterpret_cast<double2*>(red + warp * 512 + ch * 64 + lane * 2) = part[ch];
    __syncthreads();
    double2 s = make_double2(0.0, 0.0);
#pragma unroll
    for (int wv = 0; wv < PREP_WARPS; ++wv) {
        const double2 v = *reinterpret_cast<const double2*>(red + wv * 512 + threadIdx.x * 2);
        s.x += v.x;
        s.y += v.y;
    }
    return s;
}

// block_sum of both components at once (each summed in block_sum's order); scratch holds >= 34 doubles
__device__ __forceinline__ double2 block_sum2(double2 v, double* scratch) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = (blockDim.x + 31) >> 5;
    v.x = warp_sum(v.x);
    v.y = warp_sum(v.y);
    __syncthreads();
    if (lane == 0) {
        scratch[warp] = v.x;
        scratch[16 + warp] = v.y;
    }
    __syncthreads();
    if (warp == 0) {
        double sx = lane < nw ? scratch[lane] : 0.0;
        double sy = lane < nw ? scratch[16 + lane] : 0.0;
        sx = warp_sum(sx);
        sy = warp_sum(sy);
        if (lane == 0) {
            scratch[32] = sx;
            scratch[33] = sy;
        }
    }
    __syncthreads();
    return make_double2(scratch[32], scratch[33]);
}

// The prep kernel is the first writer of a window's scalar record, which lives in the shared, never-cleared workspace:
// it zeroes v1 (written by the solver, if one follows) and the unused slots, so that no call returns stale values
__device__ __forceinline__ void clear_later_slots(double* scal) {
    scal[BP_S_V1] = 0.0;
    for (int k = BP_S_MCM_AVG + 1; k < BP_S_COUNT; ++k) scal[k] = 0.0;
}

__global__ void __launch_bounds__(PREP_THREADS, 2) window_prep_kernel(PrepParams p) {
    extern __shared__ double smem[];
    const int K = p.n_window - 1;                 // daily returns per window (F2)
    double* a_s = smem;                           // [K]
    double* w0_s = a_s + ((K + 1) & ~1);          // [ldv]
    double* red = w0_s + p.ldv;                   // [PREP_WARPS][512]
    double* scratch = red + PREP_WARPS * 512;     // [40]

    const int w = blockIdx.x;
    const int tid = threadIdx.x;
    const int N = p.n_assets;
    const int day_row = p.day_row[w];
    // resampled (weekly) windows: the last return of the window is a per-date row (price at d against the
    // previous week's close) stored apart from the shared weekly rows; K1 shared rows + 1 extra row
    const int extra_row = p.extra_row ? p.extra_row[w] : -1;
    const int K1 = extra_row >= 0 ? K - 1 : K;
    const long long r0 = (long long)day_row - K1 + 1;  // first (shared) return row of the window
    const int caps_row = p.caps_row ? p.caps_row[w] : day_row;
    double* scal = p.scal + (long long)w * BP_S_COUNT;

    double sa = 0.0, saa = 0.0;
    double2 sum[NCH], wsum[NCH];
    if (p.use_band) {
        // t, p (and sum a) were produced by the banded-GEMM form of this pass (band_prep.cu)
        sa = p.band_stats[2 * (long long)w];
    } else {
    // ---- a_k = (1 + rf)^(gbar/365) - 1  (:40-48); gbar = calendar span / (n-1)
    const double gbar = (double)p.span_days[w] / (double)K;
    const double expo = gbar / 365.0;
    for (int k = tid; k < K; k += PREP_THREADS) {
        const long long rr = k < K1 ? r0 + k : (long long)extra_row;
        const double a = pow(1.0 + p.rf_row[rr], expo) - 1.0;
        a_s[k] = a;
        sa += a;
        saa = fma(a, a, saa);
    }
    sa = block_sum(sa, scratch);
    saa = block_sum(saa, scratch);

    // ---- daily column sums: t = L'1 - (sum a),  p = L'a - (a'a)/2
    for (int col0 = 0; col0 < p.ldv; col0 += 512) {
        col_accumulate<false>(p.lr_daily, p.ld, r0, K1, col0, a_s, nullptr, nullptr, false, sum, wsum);
        double2 ts = reduce_cols(sum, red);
        double2 us = reduce_cols(wsum, red);
        const int c = col0 + tid * 2;
        if (c < p.ldv && extra_row >= 0) {
            const double2 x = *reinterpret_cast<const double2*>(p.lr_daily + (long long)extra_row * p.ld + c);
            ts.x += x.x;
            ts.y += x.y;
            us.x = fma(a_s[K1], x.x, us.x);
            us.y = fma(a_s[K1], x.y, us.y);
        }
        if (c < p.ldv) {
            double2 tv = make_double2(c < N ? ts.x - sa : 0.0, c + 1 < N ? ts.y - sa : 0.0);
            double2 pv = make_double2(c < N ? us.x - 0.5 * saa : 0.0, c + 1 < N ? us.y - 0.5 * saa : 0.0);
            *reinterpret_cast<double2*>(p.t + (long long)w * p.ldv + c) = tv;
            *reinterpret_cast<double2*>(p.pvec + (long long)w * p.ldv + c) = pv;
            if (p.mode == BP_MODE_JEFFREYS) {
                *reinterpret_cast<double2*>(p.gvec + (long long)w * p.ldv + c) = tv;
                *reinterpret_cast<double2*>(p.rhs + (long long)w * p.ldv + c) = tv;
            }
        }
    }
    }
    if (p.mode == BP_MODE_JEFFREYS) {
        if (tid == 0) {
            scal[BP_S_N0] = 0.0;
            scal[BP_S_N1] = 0.0;
            scal[BP_S_ALPHA] = 0.0;
            scal[BP_S_BETA] = 1.0 / (double)(p.beta_den > 0 ? p.beta_den : p.n_window);     // J = T - (1/n) t t'  (:600)
            scal[BP_S_C] = 0.0;
            scal[BP_S_V0] = 0.0;
            scal[BP_S_M] = 0.0;
            scal[BP_S_SUMA] = sa;
            scal[BP_S_MCM_AVG] = 0.0;
            clear_later_slots(scal);
        }
        return;
    }

    // ---- MCM scaling (:90-114, :247-282): mean of the last n observations incl. d
    double avg = 0.0, n0;
    if (p.prior_n) {
        n0 = p.prior_n[w];                    // conjugate_prior_n= injection of the reference API
    } else {
        const double* mcm = p.mcm;
        const int rows = p.mcm_rows;          // min(n, available observations): iloc[-n:] semantics (:112)
        double ms = 0.0;
        // resampled windows: rows-1 shared (weekly) observations ending at day_row + the value at the trade date
        const int shared = extra_row >= 0 ? rows - 1 : rows;
        for (int k = tid; k < shared; k += PREP_THREADS) ms += mcm[day_row - shared + 1 + k];
        ms = block_sum(ms, scratch);
        const double cur = mcm[extra_row >= 0 ? extra_row : day_row];
        if (extra_row >= 0) ms += cur;
        avg = ms / (double)rows;
        const double frac = cur > avg ? cur / avg : avg / cur;
        n0 = (double)p.n_window * frac * p.mcm_scaling;
    }
    const double n1 = n0 + (double)p.n_window;

    // ---- prior weights w0 (:679-701 value weighted, :661-677 equally weighted)
    double cs = 0.0;
    if (p.prior_kind == BP_PRIOR_VW) {
        for (int j = tid; j < N; j += PREP_THREADS) cs += p.caps[(long long)caps_row * p.ld_caps + j];
        cs = block_sum(cs, scratch);
    }
    for (int j = tid; j < p.ldv; j += PREP_THREADS) {
        double v = 0.0;
        if (j < N) v = p.prior_kind == BP_PRIOR_VW ? p.caps[(long long)caps_row * p.ld_caps + j] / cs : 1.0 / (double)N;
        w0_s[j] = v;
        p.w0[(long long)w * p.ldv + j] = v;
    }
    __syncthreads();

    // HF returns of the window: m = the kept rows of the span (dropna, :314).  A dropped row is a zero row of lr_hf, so
    // every sum below may run over the whole span; only the mean divides by m and only kept rows are centred.
    const int span = p.hf_span[w];
    const long long h0 = (long long)p.hf_row0[w];           // first HF return row (first bar dropped, F5)
    const unsigned char* keep = p.hf_keep + h0;
    auto count_kept = [&]() {
        double kept = 0.0;
        for (int k = tid; k < span; k += PREP_THREADS) kept += (double)keep[k];
        return (int)block_sum(kept, scratch);
    };
    // m < 2: pandas' cov is all NaN (:317), so S0 and everything derived from it is NaN and the solve reports a pivot
    auto alpha_of = [&](int m) { return m >= 2 ? n0 * ((double)m / (double)(m - 1)) : nan(""); };   // S0 = n0 * cov * m  (:317-318, :333)
    if (p.hf_presum) {
        const int m = count_kept();
        const double alpha = alpha_of(m);
        // pre-summed day blocks: the window's column sums are <= 3 scanned vectors (suffix' + whole chunk + prefix);
        // S0 w0, v0, c and rhs follow the Gram launch (conj_post_kernel)
        const int* ids = p.hf_vids + 3 * (long long)w;
        for (int c = tid * 2; c < p.ldv; c += 2 * PREP_THREADS) {
            double2 hs = make_double2(0.0, 0.0);
#pragma unroll
            for (int k = 0; k < 3; ++k) {
                if (ids[k] >= 0) {
                    const double2 v = *reinterpret_cast<const double2*>(p.hf_vsum + (long long)ids[k] * p.ld + c);
                    hs.x += v.x;
                    hs.y += v.y;
                }
            }
            double2 hb = make_double2(c < N ? hs.x / (double)m : 0.0, c + 1 < N ? hs.y / (double)m : 0.0);
            *reinterpret_cast<double2*>(p.gvec + (long long)w * p.ldv + c) = hb;
        }
        if (tid == 0) {
            scal[BP_S_N0] = n0;
            scal[BP_S_N1] = n1;
            scal[BP_S_ALPHA] = alpha;
            scal[BP_S_BETA] = alpha * (double)m;
            scal[BP_S_C] = 0.0;
            scal[BP_S_V0] = 0.0;
            scal[BP_S_M] = (double)m;
            scal[BP_S_SUMA] = sa;
            scal[BP_S_MCM_AVG] = avg;
            clear_later_slots(scal);
        }
        return;
    }

    // ---- HF pass 1: column means hbar and row dots y_k = h_k . w0   (:314-318)
    double* y = p.y_ws + (long long)w * p.y_stride;
    const bool one_pass = p.ldv <= 512;
    int m = one_pass ? 0 : count_kept();     // one pass: counted with the sum of y below (one reduction fewer)
    double2 hs1 = make_double2(0.0, 0.0), q1 = make_double2(0.0, 0.0);
    if (one_pass) {
        hf_single_pass(p.lr_hf, p.ld, h0, span, w0_s, y, sum, wsum);
        hs1 = reduce_cols(sum, red);
        q1 = reduce_cols(wsum, red);
    } else {
        for (int col0 = 0; col0 < p.ldv; col0 += 512) {
            col_accumulate<true>(p.lr_hf, p.ld, h0, span, col0, nullptr, w0_s, y, col0 > 0, sum, wsum);
            const double2 hs = reduce_cols(sum, red);
            const int c = col0 + tid * 2;
            if (c < p.ldv) {
                double2 hb = make_double2(c < N ? hs.x / (double)m : 0.0, c + 1 < N ? hs.y / (double)m : 0.0);
                *reinterpret_cast<double2*>(p.gvec + (long long)w * p.ldv + c) = hb;
            }
        }
    }
    __syncthreads();
    // centre y over the kept rows:  y_c = y - mean(y)   (sum_k y_c = 0 => S0 w0 = alpha * H' y_c, v0 = alpha * |y_c|^2).
    // A dropped row has y = 0 and stays 0, so it enters neither the mean nor |y_c|^2 (and H' y_c, its H row being 0).
    double ys = 0.0, kept = 0.0;
    for (int k = tid; k < span; k += PREP_THREADS) {
        ys += y[k];
        kept += (double)keep[k];
    }
    if (one_pass) {
        const double2 s2 = block_sum2(make_double2(ys, kept), scratch);
        ys = s2.x;
        m = (int)s2.y;
        const int c = tid * 2;
        if (c < p.ldv) {
            double2 hb = make_double2(c < N ? hs1.x / (double)m : 0.0, c + 1 < N ? hs1.y / (double)m : 0.0);
            *reinterpret_cast<double2*>(p.gvec + (long long)w * p.ldv + c) = hb;
        }
    } else {
        ys = block_sum(ys, scratch);
    }
    const double alpha = alpha_of(m);
    const double ybar = ys / (double)m;
    double yy = 0.0;
    for (int k = tid; k < span; k += PREP_THREADS) {
        const double v = keep[k] ? y[k] - ybar : 0.0;
        if (!one_pass) y[k] = v;
        yy = fma(v, v, yy);
    }
    yy = block_sum(yy, scratch);      // block_sum's barriers also publish the centred y to the block

    const double v0 = alpha * yy;
    const double kk = n0 + (double)N + 2.0;
    const double cc = (2.0 * n0) / (kk + sqrt(kk * kk + 4.0 * n0 * v0));   // :415-418

    // ---- q = H' y_c ;  b = c * S0 w0 + t   (:489)
    if (one_pass) {
        const int c = tid * 2;
        if (c < p.ldv) {
            const double2 qs = make_double2(fma(-ybar, hs1.x, q1.x), fma(-ybar, hs1.y, q1.y));
            const double2 tv = *reinterpret_cast<const double2*>(p.t + (long long)w * p.ldv + c);
            double2 s0w0 = make_double2(c < N ? alpha * qs.x : 0.0, c + 1 < N ? alpha * qs.y : 0.0);
            double2 bv = make_double2(c < N ? fma(cc, s0w0.x, tv.x) : 0.0, c + 1 < N ? fma(cc, s0w0.y, tv.y) : 0.0);
            *reinterpret_cast<double2*>(p.s0w0 + (long long)w * p.ldv + c) = s0w0;
            *reinterpret_cast<double2*>(p.rhs + (long long)w * p.ldv + c) = bv;
        }
    } else {
        // HF pass 2
        for (int col0 = 0; col0 < p.ldv; col0 += 512) {
            col_accumulate<false>(p.lr_hf, p.ld, h0, span, col0, y, nullptr, nullptr, false, sum, wsum);
            const double2 qs = reduce_cols(wsum, red);
            const int c = col0 + tid * 2;
            if (c < p.ldv) {
                const double2 tv = *reinterpret_cast<const double2*>(p.t + (long long)w * p.ldv + c);
                double2 s0w0 = make_double2(c < N ? alpha * qs.x : 0.0, c + 1 < N ? alpha * qs.y : 0.0);
                double2 bv = make_double2(c < N ? fma(cc, s0w0.x, tv.x) : 0.0, c + 1 < N ? fma(cc, s0w0.y, tv.y) : 0.0);
                *reinterpret_cast<double2*>(p.s0w0 + (long long)w * p.ldv + c) = s0w0;
                *reinterpret_cast<double2*>(p.rhs + (long long)w * p.ldv + c) = bv;
            }
        }
    }
    if (tid == 0) {
        scal[BP_S_N0] = n0;
        scal[BP_S_N1] = n1;
        scal[BP_S_ALPHA] = alpha;
        scal[BP_S_BETA] = alpha * (double)m;     // S0 = alpha * (H'H - m hbar hbar')
        scal[BP_S_C] = cc;
        scal[BP_S_V0] = v0;
        scal[BP_S_M] = (double)m;
        scal[BP_S_SUMA] = sa;
        scal[BP_S_MCM_AVG] = avg;
        clear_later_slots(scal);
    }
}

size_t prep_smem_bytes(int n_window, int ldv) {
    const int K = n_window - 1;
    return sizeof(double) * (size_t)(((K + 1) & ~1) + ldv + PREP_WARPS * 512 + 40);
}

cudaError_t launch_window_prep(const PrepParams& p, int n_windows, cudaStream_t st, long long n_daily_rows) {
    if (n_windows <= 0) return cudaSuccess;
    if (p.use_band) {
        cudaError_t eb = launch_daily_band(p, n_windows, n_daily_rows, st);
        if (eb != cudaSuccess || p.mode == BP_MODE_JEFFREYS) return eb;      // Jeffreys needs nothing else
    }
    const size_t smem = prep_smem_bytes(p.n_window, p.ldv);
    cudaError_t e = cudaFuncSetAttribute(window_prep_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    window_prep_kernel<<<n_windows, PREP_THREADS, smem, st>>>(p);
    return cudaGetLastError();
}

// ------------------------------------------------------------------------------------------------
// Padded lower-triangular device layout [rowsS][ldS]  ->  dense symmetric [N][N]
__global__ void unpack_sym_kernel(const double* __restrict__ S, long long win_stride, int ldS, int N,
                                  double* __restrict__ out) {
    const int w = blockIdx.y;
    const double* s = S + (long long)w * win_stride;
    double* o = out + (long long)w * N * N;
    const long long total = (long long)N * N;
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total;
         i += (long long)gridDim.x * blockDim.x) {
        const int r = int(i / N), c = int(i - (long long)r * N);
        o[i] = r >= c ? s[(long long)r * ldS + c] : s[(long long)c * ldS + r];
    }
}

void launch_unpack_sym(const double* S, long long win_stride, int ldS, int N, int W, double* out, cudaStream_t st) {
    if (W <= 0) return;
    long long total = (long long)N * N;
    int bx = (int)((total + 255) / 256);
    if (bx > 256) bx = 256;
    dim3 grid(bx, W);
    unpack_sym_kernel<<<grid, 256, 0, st>>>(S, win_stride, ldS, N, out);
}

// Strided [W][ldv] vectors -> dense [W][N]
__global__ void unpack_vec_kernel(const double* __restrict__ v, int ldv, int N, long long W, double* __restrict__ out) {
    const long long total = W * N;
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total;
         i += (long long)gridDim.x * blockDim.x) {
        const long long w = i / N;
        const int c = int(i - w * N);
        out[i] = v[w * ldv + c];
    }
}

void launch_unpack_vec(const double* v, int ldv, int N, long long W, double* out, cudaStream_t st) {
    if (W <= 0) return;
    long long total = W * N;
    long long blocks = (total + 255) / 256;
    if (blocks > 4096) blocks = 4096;
    unpack_vec_kernel<<<(unsigned)blocks, 256, 0, st>>>(v, ldv, N, W, out);
}

// ------------------------------------------------------------------------------------------------
// Resampled (weekly) windows (:106, :153): out[i] = ln(P[num[i]] / P[den[i]]) for arbitrary row pairs of the
// dense daily price matrix: one row per week (week close against the previous week's close) followed by one
// row per trading date (price at d against the previous week's close).  num == den gives a zero row.
__global__ void gather_log_returns_kernel(const double* __restrict__ P, int ld_in, const int* __restrict__ num,
                                          const int* __restrict__ den, double* __restrict__ out, int ld_out,
                                          int rows, int n_assets) {
    for (int r = blockIdx.x; r < rows; r += gridDim.x) {
        const double* pn = P + (long long)num[r] * ld_in;
        const double* pd = P + (long long)den[r] * ld_in;
        const bool zero = num[r] == den[r];
        for (int c = threadIdx.x; c < ld_out; c += blockDim.x)
            out[(long long)r * ld_out + c] = (c < n_assets && !zero) ? log(pn[c] / pd[c]) : 0.0;
    }
}

void launch_gather_log_returns(const double* P, int ld_in, const int* num, const int* den, double* out, int ld_out,
                               int rows, int n_assets, cudaStream_t st) {
    if (rows <= 0) return;
    const int blocks = rows < 4096 ? rows : 4096;
    gather_log_returns_kernel<<<blocks, 128, 0, st>>>(P, ld_in, num, den, out, ld_out, rows, n_assets);
}

// ------------------------------------------------------------------------------------------------
// Range sums of stored block tiles (Gram reuse): out[r] = sum_{b in [lo_r, hi_r)} store[b], tile by tile.  The run
// of whole blocks inside a window is the same for many consecutive windows (it changes only when a window edge
// crosses a block boundary), so it is summed once here and each window adds ONE tile instead of hi-lo tiles.
// Summation order: ascending block index (deterministic).  ranges = [lo_0, hi_0, lo_1, hi_1, ...].
__global__ void range_sum_kernel(const double* __restrict__ store, const int* __restrict__ ranges, int npairs,
                                 double* __restrict__ out) {
    const int r = blockIdx.y;
    const int lo = ranges[2 * r], hi = ranges[2 * r + 1];
    const long long per_block = (long long)npairs * (GRAM_BLOCK_TILE_DOUBLES / 2);      // double2 elements per block
    const double2* src = reinterpret_cast<const double2*>(store);
    double2* dst = reinterpret_cast<double2*>(out) + (long long)r * per_block;
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < per_block; i += (long long)gridDim.x * blockDim.x) {
        double2 acc = make_double2(0.0, 0.0);
        for (int b = lo; b < hi; ++b) {
            const double2 v = src[(long long)b * per_block + i];
            acc.x += v.x;
            acc.y += v.y;
        }
        dst[i] = acc;
    }
}

void launch_range_sum(const double* store, const int* ranges, int n_ranges, int npairs, double* out, cudaStream_t st) {
    if (n_ranges <= 0) return;
    dim3 grid(64, n_ranges);
    range_sum_kernel<<<grid, 256, 0, st>>>(store, ranges, npairs, out);
}

// Columns of a window staged in shared memory at a time: 48 KB, the dynamic shared memory a launch gets without opting in
constexpr int GATHER_COL_CHUNK = 12288;

// Working market gathered from the resident pool (bp_select_market, bp_select_windows): block w = pool rows [rows[3w],
// rows[3w] + rows[3w+2]) of its own columns cols[w][0..n) (cols == nullptr: columns 0..n-1), written densely from
// working row rows[3w+1] on.  One CTA per (window, slice of rows); the window's column list sits in shared memory, in
// chunks of GATHER_COL_CHUNK columns (one chunk up to that width).  A thread keeps one column (and, for a chunk narrower
// than the CTA, one of the blockDim / nc rows handled per step), so the loop has no index division, and each step
// stores a contiguous run of the output.  HBM bound; the reads of a row are scattered over its 128-byte lines.
__global__ void gather_window_blocks_kernel(const double* __restrict__ src, long long ld_src, double* __restrict__ dst,
                                            int n, const int* __restrict__ cols, const long long* __restrict__ rows,
                                            int slice_rows) {
    extern __shared__ int wcols[];
    const int w = blockIdx.x;
    const long long s0 = rows[3 * (long long)w], d0 = rows[3 * (long long)w + 1], nr = rows[3 * (long long)w + 2];
    for (int c0 = 0; c0 < n; c0 += GATHER_COL_CHUNK) {
        const int nc = n - c0 < GATHER_COL_CHUNK ? n - c0 : GATHER_COL_CHUNK;
        if (c0 > 0) __syncthreads();                         // every thread is done with the previous chunk
        for (int j = threadIdx.x; j < nc; j += blockDim.x) wcols[j] = cols ? cols[(long long)w * n + c0 + j] : c0 + j;
        __syncthreads();
        const bool wide = nc >= (int)blockDim.x;
        const int per_step = wide ? 1 : blockDim.x / nc;     // rows per step
        const int tr = wide ? 0 : threadIdx.x / nc;          // this thread's row within a step
        const int tc = wide ? threadIdx.x : threadIdx.x % nc; // and its first column
        const int cstep = wide ? blockDim.x : nc;
        if (tr >= per_step) continue;
        for (long long r0 = (long long)blockIdx.y * slice_rows; r0 < nr; r0 += (long long)gridDim.y * slice_rows) {
            const long long r1 = nr - r0 < slice_rows ? nr : r0 + slice_rows;
            for (long long r = r0 + tr; r < r1; r += per_step) {
                const double* s = src + (s0 + r) * ld_src;
                double* d = dst + (d0 + r) * n + c0;
                for (int j = tc; j < nc; j += cstep) d[j] = s[wcols[j]];
            }
        }
    }
}

void launch_gather_window_blocks(const double* src, long long ld_src, double* dst, int n, int n_windows, const int* cols,
                                 const long long* rows, long long max_rows, cudaStream_t st) {
    if (n_windows <= 0 || n <= 0 || max_rows <= 0) return;
    const int slice_rows = n >= 2048 ? 1 : 2048 / n;
    const long long slices = (max_rows + slice_rows - 1) / slice_rows;
    const dim3 grid(n_windows, (unsigned)(slices < 65535 ? slices : 65535));
    const size_t smem = sizeof(int) * (size_t)(n < GATHER_COL_CHUNK ? n : GATHER_COL_CHUNK);
    gather_window_blocks_kernel<<<grid, 256, smem, st>>>(src, ld_src, dst, n, cols, rows, slice_rows);
}

// dst row (dst_row0 + k) = src row src_rows[k], k in [k0, k1): the overnight returns of arbitrary day blocks, gathered
// behind the intraday matrix so that a window reads them as one contiguous run (PhasePlan::inner)
__global__ void gather_rows_indexed_kernel(double* __restrict__ M, int ld, const int* __restrict__ src_rows,
                                           long long dst_row0, int k0, int k1) {
    const int k = k0 + blockIdx.x;
    if (k >= k1) return;
    const double2* src = reinterpret_cast<const double2*>(M + (long long)src_rows[k] * ld);
    double2* dst = reinterpret_cast<double2*>(M + (dst_row0 + k) * ld);
    for (int c = threadIdx.x; c < ld / 2; c += blockDim.x) dst[c] = src[c];
}

void launch_gather_rows_indexed(double* M, int ld, const int* src_rows, long long dst_row0, int k0, int k1,
                                cudaStream_t st) {
    if (k1 <= k0) return;
    gather_rows_indexed_kernel<<<k1 - k0, 128, 0, st>>>(M, ld, src_rows, dst_row0, k0, k1);
}

// ------------------------------------------------------------------------------------------------
// Pre-summed intraday day blocks (long HF look-backs).  A window of D trading days is
//   inner(first day) + FD(day 2) + ... + FD(day D),   FD(b) = inner(b) + overnight(b) (x) overnight(b)
// (inner = the day without its first, overnight, return; the window's own first bar has no return, F5).  With the
// days cut into chunks of C consecutive blocks (C = the shortest run of full days of any window) and, per chunk,
//   prefix[b]  = FD[chunk start] + ... + FD[b]               suffix'[b] = inner[b] + FD[b+1] + ... + FD[chunk end]
// every window is suffix'[first day] + (one whole chunk = prefix[chunk end])? + prefix[last day]: at most three
// stored tiles / vectors whatever the look-back, all exact FP64 sums of the same products (no subtraction).
// The same ids address the tile store (bp_api.cu) and the vector store: inner at b, suffix' at nb + b, prefix at 2nb + b.

// column sums of the inner rows of blocks [b0, b1): out[b][ld]
__global__ void block_col_sums_kernel(const double* __restrict__ M, int ld, const int* __restrict__ starts, int b0,
                                      double* __restrict__ out) {
    const int b = b0 + blockIdx.x;
    const int r0 = starts[b] + 1, r1 = starts[b + 1];
    for (int c = threadIdx.x * 2; c < ld; c += 2 * blockDim.x) {
        double2 acc = make_double2(0.0, 0.0);
        for (int r = r0; r < r1; ++r) {
            const double2 v = *reinterpret_cast<const double2*>(M + (long long)r * ld + c);
            acc.x += v.x;
            acc.y += v.y;
        }
        *reinterpret_cast<double2*>(out + (long long)b * ld + c) = acc;
    }
}

void launch_block_col_sums(const double* M, int ld, const int* starts, int b0, int b1, double* out, cudaStream_t st) {
    if (b1 <= b0) return;
    block_col_sums_kernel<<<b1 - b0, 128, 0, st>>>(M, ld, starts, b0, out);
}

// vsum rows [0, nb) hold the inner column sums; writes suffix' rows at nb + b and prefix rows at 2 nb + b
__global__ void vec_scan_kernel(double* __restrict__ vsum, int ld, const double* __restrict__ M,
                                const int* __restrict__ starts, int nb, int chunk) {
    const int c = (blockIdx.x * blockDim.x + threadIdx.x) * 2;
    if (c >= ld) return;
    const int lo = blockIdx.y * chunk, hi = min(lo + chunk, nb);
    double2 acc = make_double2(0.0, 0.0);
    for (int b = lo; b < hi; ++b) {
        const double2 in = *reinterpret_cast<const double2*>(vsum + (long long)b * ld + c);
        const double2 o = b > 0 ? *reinterpret_cast<const double2*>(M + (long long)starts[b] * ld + c) : make_double2(0.0, 0.0);
        acc.x += in.x + o.x;
        acc.y += in.y + o.y;
        *reinterpret_cast<double2*>(vsum + (long long)(2 * nb + b) * ld + c) = acc;
    }
    acc = make_double2(0.0, 0.0);
    for (int b = hi - 1; b >= lo; --b) {
        const double2 in = *reinterpret_cast<const double2*>(vsum + (long long)b * ld + c);
        const double2 o = b > 0 ? *reinterpret_cast<const double2*>(M + (long long)starts[b] * ld + c) : make_double2(0.0, 0.0);
        *reinterpret_cast<double2*>(vsum + (long long)(nb + b) * ld + c) = make_double2(in.x + acc.x, in.y + acc.y);
        acc.x += in.x + o.x;
        acc.y += in.y + o.y;
    }
}

void launch_vec_scan(double* vsum, int ld, const double* M, const int* starts, int nb, int chunk, cudaStream_t st) {
    if (nb <= 0) return;
    dim3 grid((ld / 2 + 127) / 128, (nb + chunk - 1) / chunk);
    vec_scan_kernel<<<grid, 128, 0, st>>>(vsum, ld, M, starts, nb, chunk);
}

// Tile version: store tiles [0, nb) x npairs hold the inner Gram tiles (fragment-major, as written by the block
// precompute of gram_dmma_kernel); one thread per double2 of a tile, sequential over the blocks of its chunk.
// Element (q, t) of a tile, q = 4 mt + nt, t = thread of the Gram CTA: row 128 ti + 64 (warp & 1) + 8 mt + g,
// columns 128 tj + 32 (warp >> 1) + 8 nt + 2 tig (+1).
__global__ void __launch_bounds__(256) tile_scan_kernel(double* __restrict__ store, int npairs, const double* __restrict__ M,
                                                        int ld, const int* __restrict__ starts, int nb, int chunk) {
    const int idx2 = blockIdx.x * blockDim.x + threadIdx.x;      // double2 index inside the tile, < 8192
    const int pair = blockIdx.y;
    const int lo = blockIdx.z * chunk, hi = min(lo + chunk, nb);
    int ti = 0;
    while ((ti + 1) * (ti + 2) / 2 <= pair) ++ti;
    const int tj = pair - ti * (ti + 1) / 2;
    const int q = idx2 >> 8, t = idx2 & 255;
    const int warp = t >> 5, lane = t & 31, g = lane >> 2, tig = lane & 3;
    const int i = ti * GRAM_TILE + (warp & 1) * 64 + (q >> 2) * 8 + g;
    const int j = tj * GRAM_TILE + (warp >> 1) * 32 + (q & 3) * 8 + 2 * tig;
    const bool in_i = i < ld, in_j = j < ld;                      // ld is even: j + 1 < ld whenever j < ld
    const long long tile2 = GRAM_BLOCK_TILE_DOUBLES / 2;
    double2* S = reinterpret_cast<double2*>(store);
    auto at = [&](long long id) { return S + (id * npairs + pair) * tile2 + idx2; };
    auto rank1 = [&](int b) {
        double2 r = make_double2(0.0, 0.0);
        if (b > 0 && in_i && in_j) {
            const double* o = M + (long long)starts[b] * ld;
            const double oi = o[i];
            const double2 oj = *reinterpret_cast<const double2*>(o + j);
            r.x = oi * oj.x;
            r.y = oi * oj.y;
        }
        return r;
    };
    double2 acc = make_double2(0.0, 0.0);
    for (int b = lo; b < hi; ++b) {
        const double2 in = *at(b);
        const double2 r = rank1(b);
        acc.x += in.x + r.x;
        acc.y += in.y + r.y;
        *at(2LL * nb + b) = acc;
    }
    acc = make_double2(0.0, 0.0);
    for (int b = hi - 1; b >= lo; --b) {
        const double2 in = *at(b);
        const double2 r = rank1(b);
        *at((long long)nb + b) = make_double2(in.x + acc.x, in.y + acc.y);
        acc.x += in.x + r.x;
        acc.y += in.y + r.y;
    }
}

void launch_tile_scan(double* store, int npairs, int n_tiles_side, const double* M, int ld, const int* starts, int nb,
                      int chunk, cudaStream_t st) {
    (void)n_tiles_side;
    if (nb <= 0) return;
    dim3 grid(GRAM_BLOCK_TILE_DOUBLES / 2 / 256, npairs, (nb + chunk - 1) / chunk);
    tile_scan_kernel<<<grid, 256, 0, st>>>(store, npairs, M, ld, starts, nb, chunk);
}

// S0 w0, v0, c, rhs from the Gram kernel's mat-vec partials (see PostParams)
__global__ void __launch_bounds__(256) conj_post_kernel(PostParams p) {
    __shared__ double scratch[40];
    const int w = blockIdx.x, tid = threadIdx.x;
    const int N = p.n_assets;
    const int nt = (N + GRAM_TILE - 1) / GRAM_TILE;
    const int npairs = nt * (nt + 1) / 2;
    const double* part = p.mv_part + (long long)w * npairs * 256;
    const double* w0 = p.w0 + (long long)w * p.ldv;
    const double* hb = p.gvec + (long long)w * p.ldv;
    double* scal = p.scal + (long long)w * BP_S_COUNT;
    const double n0 = scal[BP_S_N0], alpha = scal[BP_S_ALPHA], m = scal[BP_S_M];
    double hw = 0.0;
    for (int i = tid; i < N; i += 256) hw = fma(hb[i], w0[i], hw);
    hw = block_sum(hw, scratch);                                   // hbar'w0
    double v0p = 0.0;
    for (int i = tid; i < p.ldv; i += 256) {
        double s0 = 0.0;
        if (i < N) {
            const int ti = i / GRAM_TILE, k = i % GRAM_TILE;
            double raw = 0.0;
            for (int tj = 0; tj <= ti; ++tj) raw += part[((ti * (ti + 1) / 2 + tj) * 2 + 0) * 128 + k];        // tiles of row ti
            for (int tk = ti + 1; tk < nt; ++tk) raw += part[((tk * (tk + 1) / 2 + ti) * 2 + 1) * 128 + k];    // tiles of column ti
            s0 = alpha * fma(-m * hw, hb[i], raw);                // S0 w0 = alpha (G w0 - m hbar (hbar'w0))
            v0p = fma(w0[i], s0, v0p);
        }
        p.s0w0[(long long)w * p.ldv + i] = s0;
    }
    const double v0 = block_sum(v0p, scratch);
    const double kk = n0 + (double)N + 2.0;
    const double cc = (2.0 * n0) / (kk + sqrt(kk * kk + 4.0 * n0 * v0));   // :415-418
    for (int i = tid; i < p.ldv; i += 256)
        p.rhs[(long long)w * p.ldv + i] = i < N ? fma(cc, p.s0w0[(long long)w * p.ldv + i], p.t[(long long)w * p.ldv + i]) : 0.0;
    if (tid == 0) {
        scal[BP_S_C] = cc;
        scal[BP_S_V0] = v0;
    }
}

cudaError_t launch_conj_post(const PostParams& p, cudaStream_t st) {
    if (p.n_windows <= 0) return cudaSuccess;
    conj_post_kernel<<<p.n_windows, 256, 0, st>>>(p);
    return cudaGetLastError();
}

// One tile per distinct RUN TRIPLE (coarse run + fine run on the head side + fine run on the tail side): the three
// pre-summed run tiles of a window's daily rows are added up once per distinct triple (it changes only when a
// window edge crosses a fine-block boundary), so a window adds ONE tile per output tile instead of three.
// triples = [coarse_id, fineA_id, fineB_id] per output, -1 = absent.  Order: coarse + fineA + fineB (deterministic).
__global__ void combine_runs_kernel(const double* __restrict__ rs_coarse, const double* __restrict__ rs_fine,
                                    const int* __restrict__ triples, int npairs, double* __restrict__ out) {
    const int r = blockIdx.y;
    const int ic = triples[3 * r], ia = triples[3 * r + 1], ib = triples[3 * r + 2];
    const long long per_block = (long long)npairs * (GRAM_BLOCK_TILE_DOUBLES / 2);
    const double2* sc = reinterpret_cast<const double2*>(rs_coarse);
    const double2* sf = reinterpret_cast<const double2*>(rs_fine);
    double2* dst = reinterpret_cast<double2*>(out) + (long long)r * per_block;
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < per_block; i += (long long)gridDim.x * blockDim.x) {
        double2 acc = make_double2(0.0, 0.0);
        if (ic >= 0) acc = sc[(long long)ic * per_block + i];
        if (ia >= 0) {
            const double2 v = sf[(long long)ia * per_block + i];
            acc.x += v.x;
            acc.y += v.y;
        }
        if (ib >= 0) {
            const double2 v = sf[(long long)ib * per_block + i];
            acc.x += v.x;
            acc.y += v.y;
        }
        dst[i] = acc;
    }
}

void launch_combine_runs(const double* rs_coarse, const double* rs_fine, const int* triples, int n, int npairs,
                         double* out, cudaStream_t st) {
    if (n <= 0) return;
    dim3 grid(64, n);
    combine_runs_kernel<<<grid, 256, 0, st>>>(rs_coarse, rs_fine, triples, npairs, out);
}

// ------------------------------------------------------------------------------------------------
// Window descriptors travel host -> device through a page-locked host buffer read by this kernel (zero-copy
// over PCIe) instead of a cudaMemcpy: the host->device copy engine may be busy for tens of milliseconds with
// the intraday block, and a queued 80 KB descriptor copy would stall every stage that does not even read it.
__global__ void fetch_ints_kernel(const int* __restrict__ src_host, int* __restrict__ dst, long long n) {
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x)
        dst[i] = src_host[i];
}

void launch_fetch_ints(const int* src_host, int* dst, long long n, cudaStream_t st) {
    if (n <= 0) return;
    long long blocks = (n + 255) / 256;
    if (blocks > 256) blocks = 256;
    fetch_ints_kernel<<<(unsigned)blocks, 256, 0, st>>>(src_host, dst, n);
}

// ------------------------------------------------------------------------------------------------
// calculate_excess_log_returns_from_prices (:31-62) for ONE window: X[k][j] = L[r0+k][j] - a_k
__global__ void excess_returns_kernel(const double* __restrict__ lr, int ld, const double* __restrict__ rf_row,
                                      int day_row, int span_days, int n_window, int N, double* __restrict__ X) {
    const int K = n_window - 1;
    const long long r0 = (long long)day_row - K + 1;
    const double expo = ((double)span_days / (double)K) / 365.0;
    for (int k = blockIdx.x; k < K; k += gridDim.x) {
        const double a = pow(1.0 + rf_row[r0 + k], expo) - 1.0;
        for (int j = threadIdx.x; j < N; j += blockDim.x) X[(long long)k * N + j] = lr[(r0 + k) * ld + j] - a;
    }
}

void launch_excess_returns(const double* lr, int ld, const double* rf_row, int day_row, int span_days, int n_window,
                           int N, double* X, cudaStream_t st) {
    int blocks = n_window - 1;
    if (blocks > 1024) blocks = 1024;
    excess_returns_kernel<<<blocks, 128, 0, st>>>(lr, ld, rf_row, day_row, span_days, n_window, N, X);
}

// ------------------------------------------------------------------------------------------------
// Dense single-window stages used when a posterior moment is injected through the reference's
// optional arguments (conjugate_prior_S_df=, conjugate_c=, ... :382-577).  One CTA; N^2 work.
//   s0w0 = S0 w0, v0 = w0'S0w0 (:78), c (:415-418) unless given, b = c s0w0 + t (:489),
//   S1 = S0 + T (:358) unless given; S1 is written in the padded layout the solver expects.
__global__ void __launch_bounds__(256) dense_conj_prep_kernel(DenseParams p) {
    __shared__ double scratch[40];
    const int N = p.n_assets, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    double v0p = 0.0;
    for (int i = warp; i < N; i += 8) {
        double acc = 0.0;
        for (int j = lane; j < N; j += 32) acc = fma(p.S0[(long long)i * N + j], p.w0[j], acc);
        acc = warp_sum(acc);
        if (lane == 0) {
            p.s0w0[i] = acc;
            v0p = fma(p.w0[i], acc, v0p);
        }
    }
    const double v0 = block_sum(v0p, scratch);
    const double kk = p.n0 + (double)N + 2.0;
    const double cc = p.has_c ? p.c_in : (2.0 * p.n0) / (kk + sqrt(kk * kk + 4.0 * p.n0 * v0));
    if (p.T) {      // T == nullptr: only v0 and c are wanted
        for (int i = tid; i < p.ldv; i += 256) p.rhs[i] = i < N ? fma(cc, p.s0w0[i], p.t[i]) : 0.0;
        for (long long e = tid; e < (long long)N * N; e += 256) {
            const int i = int(e / N), j = int(e - (long long)i * N);
            const double v = p.S1_in ? p.S1_in[e] : p.S0[e] + p.T[e];
            p.S_out[(long long)i * p.ldS + j] = v;
        }
    }
    if (tid == 0) {
        p.scal[BP_S_N0] = p.n0;
        p.scal[BP_S_N1] = p.n1;
        p.scal[BP_S_C] = cc;
        p.scal[BP_S_V0] = v0;
    }
}

// Jeffreys dense stage: J = T - (1/n) t t' (:600-601), rhs = t
__global__ void __launch_bounds__(256) dense_jeffreys_prep_kernel(DenseParams p) {
    const int N = p.n_assets, tid = threadIdx.x;
    const double inv_n = 1.0 / (double)p.n_window;
    for (int i = tid; i < p.ldv; i += 256) p.rhs[i] = i < N ? p.t[i] : 0.0;
    for (long long e = tid; e < (long long)N * N; e += 256) {
        const int i = int(e / N), j = int(e - (long long)i * N);
        p.S_out[(long long)i * p.ldS + j] = p.T[e] - inv_n * p.t[i] * p.t[j];
    }
}

// v = w'Sw for dense S (calculate_portfolio_variance, :64-88); optionally the posterior scalars for
// an injected w1:  nu = (n1 + N + 2) w1 / (n1 - v)  (:572-575), weights = (1/gamma) nu (:836)
__global__ void __launch_bounds__(256) quadform_kernel(const double* __restrict__ S, int ldS, const double* __restrict__ w,
                                                       int N, double* v_out, double n1, double inv_gamma,
                                                       double* nu, double* weights) {
    __shared__ double scratch[40];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    double part = 0.0;
    for (int i = warp; i < N; i += 8) {
        double acc = 0.0;
        for (int j = lane; j < N; j += 32) acc = fma(S[(long long)i * ldS + j], w[j], acc);
        acc = warp_sum(acc);
        if (lane == 0) part = fma(w[i], acc, part);
    }
    const double v = block_sum(part, scratch);
    if (tid == 0) *v_out = v;
    if (nu) {
        const double mult = (n1 + (double)N + 2.0) / (n1 - v);
        for (int i = tid; i < N; i += 256) {
            nu[i] = w[i] * mult;
            weights[i] = inv_gamma * (w[i] * mult);
        }
    }
}

void launch_dense_prep(const DenseParams& p, bool jeffreys, cudaStream_t st) {
    if (jeffreys) dense_jeffreys_prep_kernel<<<1, 256, 0, st>>>(p);
    else dense_conj_prep_kernel<<<1, 256, 0, st>>>(p);
}

void launch_quadform(const double* S, int ldS, const double* w, int N, double* v_out, double n1, double inv_gamma,
                     double* nu, double* weights, cudaStream_t st) {
    quadform_kernel<<<1, 256, 0, st>>>(S, ldS, w, N, v_out, n1, inv_gamma, nu, weights);
}

}  // namespace bp
