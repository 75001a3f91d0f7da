// Jeffreys windows of CONSECUTIVE trade dates without a factorisation per window.
//
// The reference inverts J_w = T_w - t_w t_w'/n for every rebalance date (portfolio_calculations.py:600-606).  With
// x_i = l_i - a_i(w) 1 (:57) the statistic is T_w = G_w - p_w 1' - 1 p_w' with G_w the raw Gram of the window's log
// returns and p_w = L_w'a_w - (a_w'a_w)/2, and G slides exactly: G_{b+k} = G_b + sum_{i<=k} (l_new,i l_new,i' -
// l_old,i l_old,i').  Relative to the first ("base") window b of a group of G consecutive dates
//     J_{b+k} = J_b + U_k C_k U_k',   U_k = [l_new,1..k | l_old,1..k | p_{b+k} - p_b | 1 | t_{b+k} | t_b],
//     C_k = diag(+I_k, -I_k, -[0 1; 1 0], -1/n, +1/n),                                   rank 2k + 4,
// so by the Woodbury identity
//     J_{b+k}^-1 t_{b+k} = y_t - Y_k (C_k^-1 + U_k' J_b^-1 U_k)^-1 U_k' y_t,   Y_k = J_b^-1 U_k,  y_t = J_b^-1 t_{b+k}.
// Only the base window is factorised (chol_solve_kernel, J_b = L L'); this kernel solves the 30 right-hand sides of a
// group against L in one pass (Z = L^-1 R, then U'J_b^-1U = Z'Z for every pair of columns at once, then Y = L^-T Z)
// and finishes each window with a (2k+4)-dimensional elimination: 2 N^2 * 30 / (G-1) flops per window instead of
// N^3/3.  Every window is expressed relative to an exactly factorised base, never as a chain of updates, so the error
// does not grow with k.  tests/test_gpu_chain.py holds each window to the a-priori bound of tests/_chain_ref.py,
// 2 k(J_w) eta_in + 2 (k(J_b) + k(J_w)) (4 sqrt(N) + 2m + 8) u; the worst ratios to it measured on a B200 are 0.05
// (N = 1), 2e-4 (N = 31 .. 33 at the rank guard's margin) and 1.5e-6 .. 5e-7 (N = 500 .. 640).
//
// One CTA per group.  Shared memory: the right-hand-side block Y [Nr][33] (in place: R -> Z -> Y), a ring of six
// 32 x 32 factor blocks (cp.async, five blocks ahead), the 32 x 32 Gram Z'Z.  Substitutions are right-looking by 32-row panels: one warp
// solves the 32 x 32 diagonal block for all right-hand sides (lane = right-hand side, the panel column in registers),
// then all warps subtract its contribution from the remaining panels (thread = 4 rows x 1 right-hand side, the solved
// panel column in registers, factor entries as shared-memory broadcasts).
#include "common.cuh"
#include "jorion_math.cuh"
#include "kernels.h"

namespace bp {

constexpr int CG_MAX = 8;                 // windows per group (1 base + 7 chained)
constexpr int CR = 32;                    // right-hand sides (30 used)
constexpr int LDY = 33;
constexpr int CH_T = 256;
constexpr int CH_W = CH_T / 32;
// column layout of the right-hand-side block
constexpr int COL_NEW = 0, COL_OLD = 7, COL_PD = 14, COL_ONE = 21, COL_T = 22, COL_T0 = 29;
constexpr int MMAX = 2 * (CG_MAX - 1) + 4;    // 18
constexpr int NBUF = 6;                       // 32 x 32 factor blocks in flight (cp.async ring)

__device__ __forceinline__ void cp_async16_cg(void* dst, const void* src) {
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(smem_u32(dst)), "l"(src) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }

// 32 x 32 block of the factor at (row0, col0) -> dst[32][32]; rows >= N are zero-filled (the substitutions give those
// rows a zero solution and never divide by their diagonal).  Only the lower triangle of a diagonal block is read.
__device__ __forceinline__ void load_block_async(double* dst, const double* L, int ldS, int row0, int col0, int N, int tid) {
    // 256 threads x 2 chunks of 16 bytes: 32 rows x 16 chunks
#pragma unroll
    for (int q = 0; q < 2; ++q) {
        const int ch = tid + q * CH_T;          // 0..511
        const int r = ch >> 4, c2 = (ch & 15) * 2;
        double* d = dst + r * 32 + c2;
        if (row0 + r < N) cp_async16_cg(d, L + (long long)(row0 + r) * ldS + col0 + c2);
        else { d[0] = 0.0; d[1] = 0.0; }
    }
}

__global__ void __launch_bounds__(CH_T, 1) jeffreys_chain_kernel(const ChainParams p) {
    extern __shared__ __align__(16) double csm[];
    const int N = p.n_assets;
    const int Nr = (N + 31) / 32 * 32;
    const int npan = Nr / 32;
    double* Y = csm;                         // [Nr][LDY]
    double* Lb = Y + (size_t)Nr * LDY;       // [NBUF][32][32]
    double* Wm = Lb + NBUF * 32 * 32;        // [32][LDY]
    double* csol = Wm + 32 * LDY;            // [CH_W][2][32] small-system solutions (two right-hand sides)

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int g = blockIdx.x;
    const int b = g * p.group;                                   // base window
    const int gsize = min(p.group, p.n_windows - b);
    const int nb = gsize - 1;                                    // chained windows
    if (nb <= 0) return;
    const int n = p.n_window;
    const bool jorion = p.estimator == BP_EST_JORION;
    const double beta_den = jorion ? (double)(n - 1) : (double)n;      // rank-1 coefficient 1/n (:600) or 1/m (sample covariance)
    const long long day_b = p.day_row[b];
    const double* L = p.S + (long long)b * p.win_stride;

    // ---------------- right-hand sides
    for (int c = warp; c < CR; c += CH_W) {
        const double* src = nullptr;
        const double* sub = nullptr;
        double cst = 0.0;
        if (c >= COL_NEW && c < COL_NEW + 7) { if (c - COL_NEW < nb) src = p.lr_daily + (day_b + 1 + (c - COL_NEW)) * p.ld; }
        else if (c >= COL_OLD && c < COL_OLD + 7) { if (c - COL_OLD < nb) src = p.lr_daily + (day_b - n + 2 + (c - COL_OLD)) * p.ld; }
        else if (c >= COL_PD && c < COL_PD + 7) {
            if (c - COL_PD < nb) { src = p.pvec + (long long)(b + 1 + (c - COL_PD)) * p.ldv; sub = p.pvec + (long long)b * p.ldv; }
        } else if (c == COL_ONE) cst = 1.0;
        else if (c >= COL_T && c < COL_T + 7) { if (c - COL_T < nb) src = p.t + (long long)(b + 1 + (c - COL_T)) * p.ldv; }
        else if (c == COL_T0) src = p.t + (long long)b * p.ldv;
        for (int j = lane; j < Nr; j += 32) {
            double v = 0.0;
            if (j < N) v = src ? (sub ? src[j] - sub[j] : src[j]) : cst;
            Y[j * LDY + c] = v;
        }
    }
    __syncthreads();

    double z[32];
    // The factor blocks of a substitution pass are consumed in a fixed order (per panel: its diagonal block, then the
    // blocks it updates), so they are streamed through a ring of NBUF buffers with cp.async, NBUF-1 blocks ahead: the
    // loads (1-2 us from L2 / HBM each) are longer than the 0.3 us a block is worked on.
    int pf_a, pf_b, pf_cnt, cons_cnt;
    // ---------------- forward substitution  L Z = R   (block order: jp = 0.., ib = jp (diagonal), jp+1 .. npan-1)
    pf_a = 0; pf_b = 0; pf_cnt = 0; cons_cnt = 0;
    auto issue_fwd = [&]() {
        if (pf_a < npan) {
            load_block_async(Lb + (pf_cnt % NBUF) * 1024, L, p.ldS, pf_b * 32, pf_a * 32, N, tid);
            if (++pf_b == npan) { ++pf_a; pf_b = pf_a; }
        }
        cp_async_commit();          // possibly empty: keeps the group count uniform
        ++pf_cnt;
    };
    for (int i = 0; i < NBUF - 1; ++i) issue_fwd();
    for (int jp = 0; jp < npan; ++jp) {
        const int j0 = jp * 32;
        for (int ib = jp; ib < npan; ++ib, ++cons_cnt) {
            cp_async_wait<NBUF - 2>();
            __syncthreads();
            issue_fwd();
            const double* B = Lb + (cons_cnt % NBUF) * 1024;
            if (ib == jp) {
                // diagonal block: right-looking substitution in registers, lane = right-hand side
                if (warp == 0) {
                    const double rdl = j0 + lane < N ? 1.0 / B[lane * 32 + lane] : 0.0;
#pragma unroll
                    for (int i = 0; i < 32; ++i) z[i] = Y[(j0 + i) * LDY + lane];
#pragma unroll
                    for (int i = 0; i < 32; ++i) {
                        const double zi = z[i] * __shfl_sync(0xffffffffu, rdl, i);
                        z[i] = zi;
#pragma unroll
                        for (int r = i + 1; r < 32; ++r) z[r] = fma(-B[r * 32 + i], zi, z[r]);
                    }
#pragma unroll
                    for (int i = 0; i < 32; ++i) Y[(j0 + i) * LDY + lane] = z[i];
                }
                __syncthreads();
                if (warp != 0) {
#pragma unroll
                    for (int k = 0; k < 32; ++k) z[k] = Y[(j0 + k) * LDY + lane];
                }
            } else {
                double acc[4] = {0.0, 0.0, 0.0, 0.0};
#pragma unroll
                for (int k = 0; k < 32; k += 2) {
#pragma unroll
                    for (int r = 0; r < 4; ++r) {
                        const double2 l2 = *reinterpret_cast<const double2*>(B + (4 * warp + r) * 32 + k);
                        acc[r] = fma(l2.x, z[k], acc[r]);
                        acc[r] = fma(l2.y, z[k + 1], acc[r]);
                    }
                }
#pragma unroll
                for (int r = 0; r < 4; ++r) Y[(ib * 32 + 4 * warp + r) * LDY + lane] -= acc[r];
            }
        }
    }
    cp_async_wait<0>();
    __syncthreads();

    // ---------------- Wm = Z'Z: U'J^-1U for every pair of columns (and U'y_t as its columns COL_T+k)
    {
        double part[32];
#pragma unroll
        for (int a = 0; a < 32; ++a) part[a] = 0.0;
        for (int j = warp; j < N; j += CH_W) {
            const double yb = Y[j * LDY + lane];
#pragma unroll
            for (int a = 0; a < 32; ++a) part[a] = fma(Y[j * LDY + a], yb, part[a]);
        }
        // cross-warp reduction: the warps add their partial Gram into Wm one after the other
        for (int a = tid; a < 32 * LDY; a += CH_T) Wm[a] = 0.0;
        __syncthreads();
        for (int wv = 0; wv < CH_W; ++wv) {
            if (warp == wv) {
#pragma unroll
                for (int a = 0; a < 32; ++a) Wm[a * LDY + lane] += part[a];
            }
            __syncthreads();
        }
    }

    // ---------------- backward substitution  L' Y = Z   (block order: jp = npan-1.., diagonal, then the blocks of
    // row panel jp at column blocks ib = jp-1 .. 0)
    pf_a = npan - 1; pf_b = npan - 1; pf_cnt = 0; cons_cnt = 0;
    auto issue_bwd = [&]() {
        if (pf_a >= 0) {
            load_block_async(Lb + (pf_cnt % NBUF) * 1024, L, p.ldS, pf_a * 32, pf_b * 32, N, tid);
            if (--pf_b < 0) { --pf_a; pf_b = pf_a; }
        }
        cp_async_commit();
        ++pf_cnt;
    };
    for (int i = 0; i < NBUF - 1; ++i) issue_bwd();
    for (int jp = npan - 1; jp >= 0; --jp) {
        const int j0 = jp * 32;
        for (int ib = jp; ib >= 0; --ib, ++cons_cnt) {
            cp_async_wait<NBUF - 2>();
            __syncthreads();
            issue_bwd();
            const double* B = Lb + (cons_cnt % NBUF) * 1024;      // B[k][cc] = L[j0+k][ib*32+cc]
            if (ib == jp) {
                if (warp == 0) {
                    const double rdl = j0 + lane < N ? 1.0 / B[lane * 32 + lane] : 0.0;
#pragma unroll
                    for (int i = 0; i < 32; ++i) z[i] = Y[(j0 + i) * LDY + lane];
#pragma unroll
                    for (int i = 31; i >= 0; --i) {
                        const double zi = z[i] * __shfl_sync(0xffffffffu, rdl, i);
                        z[i] = zi;
#pragma unroll
                        for (int c = 0; c < i; ++c) z[c] = fma(-B[i * 32 + c], zi, z[c]);
                    }
#pragma unroll
                    for (int i = 0; i < 32; ++i) Y[(j0 + i) * LDY + lane] = z[i];
                }
                __syncthreads();
                if (warp != 0) {
#pragma unroll
                    for (int k = 0; k < 32; ++k) z[k] = Y[(j0 + k) * LDY + lane];
                }
            } else {
                double acc[4] = {0.0, 0.0, 0.0, 0.0};
#pragma unroll
                for (int k = 0; k < 32; ++k) {
                    const double2 la = *reinterpret_cast<const double2*>(B + k * 32 + 4 * warp);
                    const double2 lb = *reinterpret_cast<const double2*>(B + k * 32 + 4 * warp + 2);
                    acc[0] = fma(la.x, z[k], acc[0]);
                    acc[1] = fma(la.y, z[k], acc[1]);
                    acc[2] = fma(lb.x, z[k], acc[2]);
                    acc[3] = fma(lb.y, z[k], acc[3]);
                }
#pragma unroll
                for (int r = 0; r < 4; ++r) Y[(ib * 32 + 4 * warp + r) * LDY + lane] -= acc[r];
            }
        }
    }
    cp_async_wait<0>();
    __syncthreads();

    // ---------------- per chained window: (C^-1 + U'YU) c = U'y_t by Gauss-Jordan with partial pivoting (lane = row),
    // x = y_t - Y c, v1 = x't, weights.  Warp k-1 finishes window b+k.
    for (int k = warp + 1; k <= nb; k += CH_W) {
        const int m = 2 * k + 4;
        // column of the right-hand-side block behind row / column a of the small system, and the diagonal of C^-1
        auto col_of = [&](int a) {
            if (a < k) return COL_NEW + a;
            if (a < 2 * k) return COL_OLD + (a - k);
            if (a == 2 * k) return COL_PD + (k - 1);
            if (a == 2 * k + 1) return COL_ONE;
            if (a == 2 * k + 2) return COL_T + (k - 1);
            return COL_T0;
        };
        const int tcol = COL_T + (k - 1);
        double row[MMAX + 2];
        const bool active = lane < m;
        const int mycol = active ? col_of(lane) : 0;
#pragma unroll
        for (int c = 0; c < MMAX; ++c) {
            double v = 0.0;
            if (active && c < m) {
                v = Wm[mycol * LDY + col_of(c)];
                // C^-1
                if (c == lane) {
                    if (lane < k) v += 1.0;
                    else if (lane < 2 * k) v -= 1.0;
                    else if (lane == 2 * k + 2) v -= beta_den;
                    else if (lane == 2 * k + 3) v += beta_den;
                }
                if ((lane == 2 * k && c == 2 * k + 1) || (lane == 2 * k + 1 && c == 2 * k)) v -= 1.0;
            }
            row[c] = v;
        }
        row[MMAX] = active ? Wm[mycol * LDY + tcol] : 0.0;       // right-hand side U'y_t
        row[MMAX + 1] = active ? Wm[mycol * LDY + COL_ONE] : 0.0;    // second right-hand side U'y_1 (Jorion: C^-1 1)
        // Singularity relative to the base.  A window whose own matrix is exactly singular (an asset flat over the
        // window at a zero risk-free rate) gives a small system that is singular only in exact arithmetic: its
        // smallest pivot is 1e-21 .. 1e-19 of max |M| in floating point, never exactly 0.  Regular windows keep
        // pivots above 1e-9 of max |M| even at the rank guard's margin or with an asset flat at a positive rate
        // (cond(J) ~ 1e7; tests/test_chain_reference.py).  TAU = 2^-40 ~ 9e-13 sits orders of magnitude from both.
        double scale = 0.0;
#pragma unroll
        for (int c = 0; c < MMAX; ++c) scale = fmax(scale, fabs(row[c]));
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) scale = fmax(scale, __shfl_xor_sync(0xffffffffu, scale, o));
        const double piv_min = 0x1p-40 * scale;
        bool done = !active;
        int mypiv = -1;
        bool singular = false;
#pragma unroll
        for (int s = 0; s < MMAX; ++s) {
            if (s < m) {
                // pivot: the not yet used row with the largest |row[s]|
                double best = done ? -1.0 : fabs(row[s]);
                int bl = lane;
#pragma unroll
                for (int o = 16; o > 0; o >>= 1) {
                    const double ob = __shfl_xor_sync(0xffffffffu, best, o);
                    const int ol = __shfl_xor_sync(0xffffffffu, bl, o);
                    if (ob > best || (ob == best && ol < bl)) { best = ob; bl = ol; }
                }
                if (!(best > piv_min)) singular = true;
                const double pv = __shfl_sync(0xffffffffu, row[s], bl);
                const double f = (lane == bl || !active) ? 0.0 : row[s] / pv;
#pragma unroll
                for (int c = 0; c <= MMAX + 1; ++c) {
                    if (c > s) {
                        const double pr = __shfl_sync(0xffffffffu, row[c], bl);
                        row[c] = fma(-f, pr, row[c]);
                    }
                }
                if (lane != bl) row[s] = 0.0;
                if (lane == bl) { done = true; mypiv = s; }
            }
        }
        // solution component mypiv = rhs / pivot, held by the lane that pivoted on it
        double* cs = csol + warp * 64;            // [2][32]: solutions for the two right-hand sides
        if (active) {
            double piv = 1.0;
#pragma unroll
            for (int s = 0; s < MMAX; ++s) if (s == mypiv) piv = row[s];
            if (mypiv >= 0) {
                cs[mypiv] = row[MMAX] / piv;
                cs[32 + mypiv] = row[MMAX + 1] / piv;
            }
        }
        __syncwarp();
        const long long w = b + k;
        const double* tk = p.t + w * p.ldv;
        const int sb = p.status[b];
        if (!jorion) {
            double v1 = 0.0;
            for (int j = lane; j < p.ldv; j += 32) {
                double x = 0.0;
                if (j < N) {
                    x = Y[j * LDY + tcol];
                    for (int a = 0; a < m; ++a) x = fma(-cs[a], Y[j * LDY + col_of(a)], x);
                    v1 = fma(x, tk[j], v1);
                }
                p.w1[w * p.ldv + j] = x;
                p.nu[w * p.ldv + j] = x;
                p.weights[w * p.ldv + j] = p.inv_gamma * x;
            }
            v1 = warp_sum(v1);
            if (lane == 0) {
                p.scal[w * BP_S_COUNT + BP_S_V1] = v1;
                p.status[w] = sb != 0 ? sb : (singular || !(v1 > 0.0) ? N + 1 : 0);
            }
        } else {
            // y = C^-1 t and z = C^-1 1 of this window (kept in w1 / nu for the second pass), then the Bayes-Stein weights
            double sy = 0.0, sz = 0.0, ty = 0.0;
            for (int j = lane; j < N; j += 32) {
                double y = Y[j * LDY + tcol], z1 = Y[j * LDY + COL_ONE];
                for (int a = 0; a < m; ++a) {
                    const double ya = Y[j * LDY + col_of(a)];
                    y = fma(-cs[a], ya, y);
                    z1 = fma(-cs[32 + a], ya, z1);
                }
                p.w1[w * p.ldv + j] = y;
                p.nu[w * p.ldv + j] = z1;
                sy += y;
                sz += z1;
                ty = fma(tk[j], y, ty);
            }
            sy = warp_sum(sy);
            sz = warp_sum(sz);
            ty = warp_sum(ty);
            const JorionCoef jc = jorion_coefficients(sy, sz, ty, (double)(n - 1), (double)N);
            for (int j = lane; j < p.ldv; j += 32) {
                double nu = 0.0;
                if (j < N) nu = jc.c_y * p.w1[w * p.ldv + j] + jc.c_z * p.nu[w * p.ldv + j];     // own writes of this lane
                else p.w1[w * p.ldv + j] = 0.0;
                p.nu[w * p.ldv + j] = nu;
                p.weights[w * p.ldv + j] = p.inv_gamma * nu;
            }
            if (lane == 0) {
                double* sc = p.scal + w * BP_S_COUNT;
                sc[BP_S_JORION_MU_G] = jc.mu_g;
                sc[BP_S_JORION_LAMBDA] = jc.lambda;
                sc[BP_S_JORION_V] = jc.v;
                sc[BP_S_JORION_Q] = jc.q;
                sc[BP_S_JORION_ONE_VINV_ONE] = jc.one_vinv_one;
                p.status[w] = sb != 0 ? sb : (singular || !(ty > 0.0) ? N + 1 : 0);
            }
        }
        __syncwarp();
    }
}

size_t chain_smem_bytes(int n_assets) {
    const int Nr = (n_assets + 31) / 32 * 32;
    return sizeof(double) * ((size_t)Nr * LDY + NBUF * 32 * 32 + 32 * LDY + CH_W * 64 + 40);
}

int chain_max_group() { return CG_MAX; }

cudaError_t launch_jeffreys_chain(const ChainParams& p, cudaStream_t st) {
    if (p.n_windows <= 0 || p.group < 2) return cudaSuccess;
    if (p.group > CG_MAX) return cudaErrorInvalidValue;
    const size_t smem = chain_smem_bytes(p.n_assets);
    cudaError_t e = cudaFuncSetAttribute(jeffreys_chain_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    const int groups = (p.n_windows + p.group - 1) / p.group;
    jeffreys_chain_kernel<<<groups, CH_T, smem, st>>>(p);
    return cudaGetLastError();
}

}  // namespace bp
