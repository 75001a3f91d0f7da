// Daily column sums of consecutive windows as a BANDED GEMM on the FP64 tensor cores.
//
// Per window w the reference needs (portfolio_calculations.py:40-57, :222, F3)
//   t_w = sum_k x_k = L'1 - (sum a) 1          u_w = L'a_w         a_k(w) = (1 + rf_k)^(gbar_w/365) - 1
// over its K = n-1 daily log-return rows.  The exponent depends on the window's calendar span, so the weights
// are not shared between windows and every window used to stream its own K x N rows (window_prep_kernel:
// 16.7 GB of L2 reads per Jeffreys batch at N=500, n=1008, K=1007; 2.6 ms at 6.4 TB/s, 98.7% L2 hits).
// But consecutive rebalance dates shift the window by one row: for a tile of 32 windows the union of their rows
// is K+31 rows, and [T; U] = [B; A] L with the 64 x (K+31) band matrix (B = 0/1 band indicator, A = the weights
// inside the band) is 2 * 64 * (K+31) * N flops per tile -- 8.5 GFLOP for the whole batch, and every row of L
// is read once per 32 windows instead of once per window.
//
//   rf_weights_kernel   a_k(w), sum a, sum a^2 per window (the pow() work, as before, once per window)
//   daily_band_kernel   one CTA per (32 windows, 128 columns): rows in chunks of 32 through a double-buffered
//                       cp.async pipeline, band matrix chunk built in shared memory, mma.sync.m8n8k4.f64;
//                       epilogue t = T - sum a, p = U - (a'a)/2 (and g = rhs = t for Jeffreys)
// The products are the same as in the per-window pass (1.0 * x and a_k * x); only the summation order differs.
#include "common.cuh"
#include "kernels.h"

namespace bp {

constexpr int BAND_WT = 32;                  // windows per tile
constexpr int BAND_CT = 128;                 // columns per tile
constexpr int BAND_RC = 32;                  // rows per chunk
constexpr int BAND_LS = BAND_CT + 4;         // row stride of the L chunk (doubles): lanes (g,tig) hit bank 4 tig + g
constexpr int BAND_AS = 2 * BAND_WT + 4;     // row stride of the band chunk
constexpr int BAND_THREADS = 256;
constexpr int BAND_SMEM = 2 * BAND_RC * (BAND_LS + BAND_AS) * (int)sizeof(double);

// one CTA per window: weights into aw[w][0..K), stats[w] = {sum a, sum a^2}; Jeffreys scalars
__global__ void __launch_bounds__(128) rf_weights_kernel(PrepParams p, int K) {
    __shared__ double scratch[40];
    const int w = blockIdx.x, tid = threadIdx.x;
    const long long r0 = (long long)p.day_row[w] - K + 1;
    const double expo = ((double)p.span_days[w] / (double)K) / 365.0;      // gbar / 365  (:40-48)
    double* aw = p.band_aw + (long long)w * p.band_ld;
    double sa = 0.0, saa = 0.0;
    for (int k = tid; k < K; k += 128) {
        const double a = pow(1.0 + p.rf_row[r0 + k], expo) - 1.0;
        aw[k] = a;
        sa += a;
        saa = fma(a, a, saa);
    }
    sa = block_sum(sa, scratch);
    saa = block_sum(saa, scratch);
    if (tid == 0) {
        p.band_stats[2 * (long long)w] = sa;
        p.band_stats[2 * (long long)w + 1] = saa;
        if (p.mode == BP_MODE_JEFFREYS) {
            double* scal = p.scal + (long long)w * BP_S_COUNT;
            scal[BP_S_N0] = 0.0;
            scal[BP_S_N1] = 0.0;
            scal[BP_S_ALPHA] = 0.0;
            scal[BP_S_BETA] = 1.0 / (double)(p.beta_den > 0 ? p.beta_den : p.n_window);     // J = T - (1/n) t t'  (:600)
            scal[BP_S_C] = 0.0;
            scal[BP_S_V0] = 0.0;
            scal[BP_S_M] = 0.0;
            scal[BP_S_SUMA] = sa;
            // first writer of the record in the never-cleared workspace (see window_prep_kernel): no stale slot
            scal[BP_S_MCM_AVG] = 0.0;
            scal[BP_S_V1] = 0.0;
            for (int k = BP_S_MCM_AVG + 1; k < BP_S_COUNT; ++k) scal[k] = 0.0;
        }
    }
}

__device__ __forceinline__ void cp_async16(void* dst, const void* src, bool valid) {
    const int bytes = valid ? 16 : 0;      // src-size 0: zero fill
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(smem_u32(dst)), "l"(src), "r"(bytes) : "memory");
}

__global__ void __launch_bounds__(BAND_THREADS, 2) daily_band_kernel(PrepParams p, int K, int n_windows, long long n_rows) {
    extern __shared__ __align__(16) double band_sm[];
    double* Ls = band_sm;                                  // [2][BAND_RC][BAND_LS]
    double* As = Ls + 2 * BAND_RC * BAND_LS;               // [2][BAND_RC][BAND_AS]
    __shared__ int r0s[BAND_WT];
    __shared__ int rng[2];
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31, g = lane >> 2, tig = lane & 3;
    const int w0 = blockIdx.x * BAND_WT, col0 = blockIdx.y * BAND_CT;
    if (tid < BAND_WT) r0s[tid] = w0 + tid < n_windows ? p.day_row[w0 + tid] - K + 1 : -(1 << 29);
    __syncthreads();
    if (tid == 0) {
        int lo = 1 << 30, hi = -(1 << 30);
        for (int j = 0; j < BAND_WT; ++j)
            if (w0 + j < n_windows) {
                lo = min(lo, r0s[j]);
                hi = max(hi, r0s[j] + K);
            }
        rng[0] = lo;
        rng[1] = hi;
    }
    __syncthreads();
    const int rmin = rng[0];
    const int nch = (rng[1] - rmin + BAND_RC - 1) / BAND_RC;

    // band chunk: thread -> window j = tid/8, rows 4*(tid%8) .. +3 of the chunk
    const int aj = tid >> 3, ai0 = (tid & 7) * 4;
    const int aj_r0 = r0s[aj];
    const double* aw = p.band_aw + (long long)(w0 + aj) * p.band_ld;
    auto fill = [&](int ch, int buf) {
        const int rbase = rmin + ch * BAND_RC;
        // L chunk: 32 rows x 128 columns, 16-byte cp.async, zero fill outside the matrix
#pragma unroll
        for (int u = 0; u < BAND_RC * BAND_CT / 2 / BAND_THREADS; ++u) {
            const int idx = tid + BAND_THREADS * u;
            const int row = idx >> 6, unit = idx & 63;
            const long long r = (long long)rbase + row;
            const int c = col0 + 2 * unit;
            const bool ok = r >= 0 && r < n_rows && c < p.ld;
            cp_async16(Ls + ((size_t)buf * BAND_RC + row) * BAND_LS + 2 * unit, p.lr_daily + (ok ? r * p.ld + c : 0), ok);
        }
        asm volatile("cp.async.commit_group;" ::: "memory");
        double* Ab = As + (size_t)buf * BAND_RC * BAND_AS;
#pragma unroll
        for (int e = 0; e < 4; ++e) {
            const int k = rbase + ai0 + e - aj_r0;
            const bool inb = k >= 0 && k < K;
            Ab[(ai0 + e) * BAND_AS + aj] = inb ? 1.0 : 0.0;
            Ab[(ai0 + e) * BAND_AS + BAND_WT + aj] = inb ? aw[k] : 0.0;
        }
    };

    double acc[8][2][2];
#pragma unroll
    for (int mt = 0; mt < 8; ++mt)
#pragma unroll
        for (int nt = 0; nt < 2; ++nt) acc[mt][nt][0] = acc[mt][nt][1] = 0.0;

    if (nch > 0) fill(0, 0);
    for (int ch = 0; ch < nch; ++ch) {
        const int buf = ch & 1;
        if (ch + 1 < nch) {
            fill(ch + 1, buf ^ 1);
            asm volatile("cp.async.wait_group 1;" ::: "memory");
        } else {
            asm volatile("cp.async.wait_group 0;" ::: "memory");
        }
        __syncthreads();
        const double* Lb = Ls + (size_t)buf * BAND_RC * BAND_LS + 16 * warp + g;
        const double* Ab = As + (size_t)buf * BAND_RC * BAND_AS + g;
#pragma unroll
        for (int ks = 0; ks < BAND_RC / 4; ++ks) {
            const int row = 4 * ks + tig;
            const double b0 = Lb[row * BAND_LS], b1 = Lb[row * BAND_LS + 8];
#pragma unroll
            for (int mt = 0; mt < 8; ++mt) {
                const double a = Ab[row * BAND_AS + 8 * mt];
                dmma884(acc[mt][0][0], acc[mt][0][1], a, b0);
                dmma884(acc[mt][1][0], acc[mt][1][1], a, b1);
            }
        }
        __syncthreads();          // the buffer is refilled in the next iteration
    }

    // epilogue: m-tile mt < 4 holds the plain sums of windows 8mt+g, m-tile mt+4 the weighted sums of the same
    // windows; columns col0 + 16 warp + 8 nt + 2 tig (+1)
    const int N = p.n_assets;
#pragma unroll
    for (int mt = 0; mt < 4; ++mt) {
        const int w = w0 + 8 * mt + g;
        if (w >= n_windows) continue;
        const double sa = p.band_stats[2 * (long long)w], saa = p.band_stats[2 * (long long)w + 1];
#pragma unroll
        for (int nt = 0; nt < 2; ++nt) {
            const int c = col0 + 16 * warp + 8 * nt + 2 * tig;
            if (c >= p.ldv) continue;
            const double2 tv = make_double2(c < N ? acc[mt][nt][0] - sa : 0.0, c + 1 < N ? acc[mt][nt][1] - sa : 0.0);
            const double2 pv = make_double2(c < N ? acc[mt + 4][nt][0] - 0.5 * saa : 0.0,
                                            c + 1 < N ? acc[mt + 4][nt][1] - 0.5 * saa : 0.0);
            *reinterpret_cast<double2*>(p.t + (long long)w * p.ldv + c) = tv;
            *reinterpret_cast<double2*>(p.pvec + (long long)w * p.ldv + c) = pv;
            if (p.mode == BP_MODE_JEFFREYS) {
                *reinterpret_cast<double2*>(p.gvec + (long long)w * p.ldv + c) = tv;
                *reinterpret_cast<double2*>(p.rhs + (long long)w * p.ldv + c) = tv;
            }
        }
    }
}

// daily part of the window prep for n_windows windows with (nearly) consecutive trade dates
cudaError_t launch_daily_band(const PrepParams& p, int n_windows, long long n_rows, cudaStream_t st) {
    if (n_windows <= 0) return cudaSuccess;
    const int K = p.n_window - 1;
    rf_weights_kernel<<<n_windows, 128, 0, st>>>(p, K);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return e;
    e = cudaFuncSetAttribute(daily_band_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, BAND_SMEM);
    if (e != cudaSuccess) return e;
    dim3 grid((n_windows + BAND_WT - 1) / BAND_WT, (p.ldv + BAND_CT - 1) / BAND_CT);
    daily_band_kernel<<<grid, BAND_THREADS, BAND_SMEM, st>>>(p, K, n_windows, n_rows);
    return cudaGetLastError();
}

}  // namespace bp
