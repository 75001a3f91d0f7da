// The arithmetic shared by the two Cholesky solvers, chol_solve_kernel (chol_solve.cu, one CTA per window) and
// chol_cluster_kernel (chol_cluster.cu, one thread-block cluster per window).  A batch's weights must not depend on
// how its windows are split over launches, so both kernels run exactly these operations in exactly this order;
// only the schedule (which CTA, warp and accumulator slot handles which m-tile) and the synchronisation differ.
// The condition estimate (chol_rcond.cu) solves with the factor through the same diagonal-block and substitution code.
//
// Fragment layout: lane (g, tig) of a warp (g = lane / 4, tig = lane % 4) holds, for the 8-row m-tile that starts at
// row `row - g` of the window, acc[nt][h] = entry (row, j0 + 8 nt + 2 tig + h) of the 32-column panel j0.  Rows below
// N that are not right-hand sides, and columns from N on, are padding (is_data_row).  Every loop here that indexes a
// fragment array is unrolled, or the array goes to local memory.
#pragma once

#include "common.cuh"
#include "jorion_math.cuh"
#include "kernels.h"

namespace bp {
namespace chol {

constexpr int NB = 32;                      // panel width and back-substitution block
constexpr int LDQ = 34;                     // row stride of the packed diagonal-block array P
constexpr int BOX_BYTES = 32 * 16 * 8;      // one TMA box: 32 rows x 16 columns of doubles

__device__ __forceinline__ void tma_load_2d(void* smem_dst, const void* tmap, int c0, int c1, uint64_t* bar) {
    asm volatile(
        "cp.async.bulk.tensor.2d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];"
        ::"r"(smem_u32(smem_dst)), "l"(reinterpret_cast<uint64_t>(tmap)), "r"(c0), "r"(c1), "r"(smem_u32(bar))
        : "memory");
}
// generic-proxy global writes (the factor) must be visible to later async-proxy (TMA) reads
__device__ __forceinline__ void fence_proxy_async_all() { asm volatile("fence.proxy.async.global;" ::: "memory"); }

// Thread 0: the TMA ring's barriers (full: one arrival plus the bytes, empty: one arrival per consumer warp)
template <int NSTAGES, int NWARPS>
__device__ __forceinline__ void init_tma_ring(const void* smap, uint64_t* full_bar, uint64_t* empty_bar) {
    tma_prefetch_desc(smap);
    for (int s = 0; s < NSTAGES; ++s) {
        mbar_init(&full_bar[s], 1);
        mbar_init(&empty_bar[s], NWARPS);
    }
    fence_barrier_init();
    fence_proxy_async();
}

// Rows of the factorisation that carry data: the N rows of S and the right-hand side(s) at rows R .. R+nrhs-1
__device__ __forceinline__ bool is_data_row(int row, int N, int R, int nrhs) {
    return row < N || (row >= R && row < R + nrhs);
}

// Cholesky factor AND inverse of one 8x8 diagonal tile, by one warp, entirely in registers.
// The tile is in DMMA accumulator layout: lane (g,tig) holds D[g][2tig], D[g][2tig+1] (lower part valid).
// On return d0/d1 hold L (zero above the diagonal) and y0/y1 inv(L), same layout.  Eight steps, each one
// round of shuffles (pivot, own-row and own-column entries of column k, row k of the inverse) and a
// handful of FMAs -- the 32-step shared-memory loop this replaces cost 170 instructions per warp and step
// and was a third of the kernel.  Inverse: with Y[i][j] = inv(L)[i][j] L[i][i], Y[i][j] -= (D[i][k]/piv) Y[k][j]
// for j <= k < i; the row scaling is applied at the end.  Returns the 1-based index of the first
// non-positive pivot, or 0.
__device__ __forceinline__ int potrf8_inv8(double& d0, double& d1, double& y0, double& y1, int g, int tig, int lane) {
    constexpr unsigned FULL = 0xffffffffu;
    int fail = 0;
    double u0 = 2 * tig == g ? 1.0 : 0.0, u1 = 2 * tig + 1 == g ? 1.0 : 0.0;
    double invrow = 0.0;
#pragma unroll
    for (int k = 0; k < 8; ++k) {
        const double dk = (k & 1) ? d1 : d0;
        const int sq = k >> 1;
        const double piv = __shfl_sync(FULL, dk, 4 * k + sq);               // D[k][k]
        const double colg = __shfl_sync(FULL, dk, (lane & ~3) | sq);        // D[g][k]
        const double colj0 = __shfl_sync(FULL, dk, 8 * tig + sq);           // D[2tig][k]
        const double colj1 = __shfl_sync(FULL, dk, 8 * tig + 4 + sq);       // D[2tig+1][k]
        const double yk0 = __shfl_sync(FULL, u0, 4 * k + tig);              // Y[k][2tig]
        const double yk1 = __shfl_sync(FULL, u1, 4 * k + tig);              // Y[k][2tig+1]
        if (!(piv > 0.0) && fail == 0) fail = k + 1;
        const double inv = rsqrt(piv);
        const double lg = colg * inv;
        const double mg = lg * inv;
        if (g == k) invrow = inv;
        if (g > k) {
            if (2 * tig > k) d0 = fma(-lg, colj0 * inv, d0);
            if (2 * tig + 1 > k) d1 = fma(-lg, colj1 * inv, d1);
            if (2 * tig <= k) u0 = fma(-mg, yk0, u0);
            if (2 * tig + 1 <= k) u1 = fma(-mg, yk1, u1);
        }
        if (sq == tig) {
            if (k & 1) d1 = g >= k ? lg : 0.0;
            else d0 = g >= k ? lg : 0.0;
        }
    }
    y0 = u0 * invrow;
    y1 = u1 * invrow;
    return fail;
}

// B fragment of the panel solve: with W = L_d whose 8x8 diagonal tiles are replaced by their inverses,
// W[8nb+n][8kb+k] sits TRANSPOSED and shifted by one column in the strictly upper part of P, at
// P[(8kb+k)*LDQ + 8nb+n+1]; lanes (g,tig) read 8-byte bank (4 tig + g + const) mod 16: conflict free.
// Inside a diagonal tile the entries above the diagonal (k > n) are zero (that spot holds L itself).
__device__ __forceinline__ double wfrag(const double* P, int kb, int nb, int h, int g, int tig) {
    const double v = P[(8 * kb + 2 * tig + h) * LDQ + 8 * nb + g + 1];
    return (nb == kb && 2 * tig + h > g) ? 0.0 : v;
}

// U, start: the accumulators of one m-tile start as -S (identity rows for the padding) and then collect +L L',
// so that they end as -C.  `present`: the tile exists in this pass.  Row R of the factorisation is the right-hand
// side, row R+1 (NRHS = 2) the vector of ones.  RHS_IN_S: the caller has stored both in rows R, R+1 of S, so every
// row is read from S (chol_solve_kernel); otherwise row R is read from rhs (chol_cluster_kernel, whose CTAs would
// need a cluster barrier to share a stored copy).
template <int NRHS, bool RHS_IN_S>
__device__ __forceinline__ void tile_start(double (&acc)[4][2], int row, bool present, const double* S, int ld,
                                           const double* rhs, int N, int R, int j0, int tig) {
    const bool real = present && is_data_row(row, N, R, NRHS);
#pragma unroll
    for (int nt = 0; nt < 4; ++nt) {
        const int col = j0 + 8 * nt + 2 * tig;
        double2 sv = make_double2(0.0, 0.0);
        if (real && col < N) {
            if (RHS_IN_S || row < N) sv = *reinterpret_cast<const double2*>(S + (long long)row * ld + col);
            else if (NRHS == 2 && row == R + 1) sv = make_double2(1.0, 1.0);
            else sv = *reinterpret_cast<const double2*>(rhs + col);
        }
        if (real) {
            acc[nt][0] = -sv.x;
            acc[nt][1] = col + 1 < N ? -sv.y : 0.0;
        } else {
            acc[nt][0] = row == col ? -1.0 : 0.0;
            acc[nt][1] = row == col + 1 ? -1.0 : 0.0;
        }
    }
}

// U, end: padding rows and columns hold no data; whatever the update accumulated there is replaced by the identity.
// In a padding column that is zero for the rows of S and a unit diagonal for a right-hand-side row R < Nr, which
// sits in the diagonal block of the last panel: its pivot must not be zero.
template <int NRHS>
__device__ __forceinline__ void tile_fix_padding(double (&acc)[4][2], int row, int N, int R, int j0, int tig) {
    const bool real = is_data_row(row, N, R, NRHS);
#pragma unroll
    for (int nt = 0; nt < 4; ++nt) {
        const int col = j0 + 8 * nt + 2 * tig;
        if (!real || col >= N) acc[nt][0] = row == col ? -1.0 : 0.0;
        if (!real || col + 1 >= N) acc[nt][1] = row == col + 1 ? -1.0 : 0.0;
    }
}

// F: the 32x32 diagonal block, blocked by 8 in fragment space, by the CTA whose warp q < 4 holds row block q in
// acc (= -C of the panel's first four m-tiles).  Column block cb: warp cb factors and inverts its 8x8 tile in
// registers; the warps below solve their tile against it (2 DMMAs) and update their remaining tiles (2 DMMAs each).
// L goes to the lower part of P, W' to the upper part.  The first failing pivot of S goes to fail_s, unless an
// earlier panel set it.
__device__ __forceinline__ void factor_diag_block(double (&acc)[4][2], double* P, int& fail_s, int j0, int N,
                                                  int warp, int lane) {
    const int g = lane >> 2, tig = lane & 3;
#pragma unroll
    for (int cb = 0; cb < NB / 8; ++cb) {
        if (warp == cb) {
            double d0 = -acc[cb][0], d1 = -acc[cb][1], y0, y1;
            const int f = potrf8_inv8(d0, d1, y0, y1, g, tig, lane);
            // a tile from row N on holds padding and right-hand sides, whose pivots are none of S's
            // (a right-hand side's is 1 - |its z in this panel|^2 and may be negative)
            if (lane == 0 && f != 0 && fail_s == 0 && j0 + 8 * cb < N) fail_s = j0 + 8 * cb + f;
            double* row = P + (8 * cb + g) * LDQ + 8 * cb + 2 * tig;
            if (2 * tig <= g) row[0] = d0;
            if (2 * tig + 1 <= g) row[1] = d1;
            if (2 * tig <= g) P[(8 * cb + 2 * tig) * LDQ + 8 * cb + g + 1] = y0;
            if (2 * tig + 1 <= g) P[(8 * cb + 2 * tig + 1) * LDQ + 8 * cb + g + 1] = y1;
        }
        __syncthreads();
        if (cb == NB / 8 - 1) break;
        if (warp > cb && warp < NB / 8) {
            double x0 = 0.0, x1 = 0.0;
#pragma unroll
            for (int h = 0; h < 2; ++h) dmma884(x0, x1, acc[cb][h], wfrag(P, cb, cb, h, g, tig));
            x0 = -x0;
            x1 = -x1;
            acc[cb][0] = x0;      // this tile now holds +L
            acc[cb][1] = x1;
            double* row = P + (8 * warp + g) * LDQ + 8 * cb + 2 * tig;
            row[0] = x0;
            row[1] = x1;
            P[(8 * cb + 2 * tig) * LDQ + 8 * warp + g + 1] = x0;
            P[(8 * cb + 2 * tig + 1) * LDQ + 8 * warp + g + 1] = x1;
        }
        __syncthreads();
        if (warp > cb && warp < NB / 8) {
#pragma unroll
            for (int nb = cb + 1; nb < NB / 8; ++nb)
                if (nb <= warp) {
#pragma unroll
                    for (int h = 0; h < 2; ++h)
                        dmma884(acc[nb][0], acc[nb][1], acc[cb][h], wfrag(P, cb, nb, h, g, tig));
                }
        }
    }
}

// Writes L_d from P back to the factor (lower part, data rows only: in the last panel z of a right-hand side R < Nr)
template <int NRHS, int NWARPS>
__device__ __forceinline__ void store_diag_block(double* S, int ld, const double* P, int j0, int N, int R, int warp,
                                                 int lane) {
    for (int i = warp; i < NB; i += NWARPS) {
        const int row = j0 + i, col = j0 + lane;
        if (is_data_row(row, N, R, NRHS) && col < N && lane <= i) S[(long long)row * ld + col] = P[i * LDQ + lane];
    }
}

// T: X = C inv(L_d)' of one m-tile below the diagonal block, straight from its accumulators, by block forward
// substitution with W: X_cb = C_cb inv(L_cb,cb)', C_nb -= X_cb L_nb,cb' (nb > cb).  DMMA step h contracts the
// columns 8cb+2tig+h the lanes already hold, so the accumulators are used as A fragments as they are.  The finished
// factor row is stored once.
template <int NRHS>
__device__ __forceinline__ void tile_solve(double (&acc)[4][2], const double* P, double* S, int ld, int row, int N,
                                           int R, int j0, int g, int tig) {
    const bool real = is_data_row(row, N, R, NRHS);
#pragma unroll
    for (int cb = 0; cb < NB / 8; ++cb) {
        double x0 = 0.0, x1 = 0.0;
#pragma unroll
        for (int h = 0; h < 2; ++h) dmma884(x0, x1, acc[cb][h], wfrag(P, cb, cb, h, g, tig));
        x0 = -x0;
        x1 = -x1;
        const int col = j0 + 8 * cb + 2 * tig;
        if (real && col < N) *reinterpret_cast<double2*>(S + (long long)row * ld + col) = make_double2(x0, x1);
#pragma unroll
        for (int nb = cb + 1; nb < NB / 8; ++nb) {
            dmma884(acc[nb][0], acc[nb][1], x0, wfrag(P, cb, nb, 0, g, tig));
            dmma884(acc[nb][0], acc[nb][1], x1, wfrag(P, cb, nb, 1, g, tig));
        }
    }
}

// z = L^-1 b sits in row R (+r) of the factor: copies it to z[NRHS][Nr] (zero beyond N) and returns
// v1 = z'z = w1' S1 w1 (:574) to every thread.
template <int NRHS, int NTHREADS>
__device__ __forceinline__ double load_z(double* z, const double* S, int ld, int N, int Nr, int R, double* scratch) {
    double zz = 0.0;
    for (int j = threadIdx.x; j < Nr; j += NTHREADS) {
        const double zj = j < N ? S[(long long)R * ld + j] : 0.0;
        z[j] = zj;
        zz = fma(zj, zj, zz);
        if constexpr (NRHS == 2) z[Nr + j] = j < N ? S[(long long)(R + 1) * ld + j] : 0.0;
    }
    return block_sum(zz, scratch);
}

// Back substitution L' x = z, right-looking over the 32-column blocks b = Nr/32-1 .. 0.  Per block: the diagonal
// block goes to P (load_diag_block), warp r solves the block's triangle for right-hand side r (solve_diag_block),
// and every block bb < b is reduced by L[rows of b, columns of bb]' x_b (reduce_block, one warp per block).

// Diagonal block b of L into P[32][LDQ] (lower part; unit diagonal for the padding)
template <int NWARPS>
__device__ __forceinline__ void load_diag_block(double* P, const double* S, int ld, int b, int N, int warp, int lane) {
    const int j0 = NB * b;
    for (int i = warp; i < NB; i += NWARPS) {
        const int row = j0 + i, col = j0 + lane;
        double v;
        if (row < N && col < N) v = lane <= i ? S[(long long)row * ld + col] : 0.0;
        else v = i == lane ? 1.0 : 0.0;
        P[i * LDQ + lane] = v;
    }
}

// One warp solves L_d' x = r for the 32 entries r (lane k holds entry k) of one block; returns x the same way
__device__ __forceinline__ double solve_diag_block(double r, const double* P, int lane) {
    const double rd = 1.0 / P[lane * LDQ + lane];      // all 32 reciprocals in parallel
#pragma unroll
    for (int k = NB - 1; k >= 0; --k) {
        const double xk = __shfl_sync(0xffffffffu, r * rd, k);
        if (lane == k) r = xk;
        if (lane < k) r = fma(-P[k * LDQ + lane], xk, r);
    }
    return r;
}

// z[r][col] -= sum_i L[j0 + i][col] x[r][j0 + i] over the rows of block b (j0 = 32 b), for column col of an
// earlier block; z and x are [NRHS][Nr] and may be the same array
template <int NRHS>
__device__ __forceinline__ void reduce_block(double* z, const double* x, const double* S, int ld, int Nr, int N, int b,
                                             int col) {
    const int j0 = NB * b;
    const int rows = min(NB, N - j0);
    double a0[NRHS], a1[NRHS];
#pragma unroll
    for (int r = 0; r < NRHS; ++r) a0[r] = a1[r] = 0.0;
#pragma unroll 4
    for (int i = 0; i + 1 < rows; i += 2) {
        const double l0 = S[(long long)(j0 + i) * ld + col], l1 = S[(long long)(j0 + i + 1) * ld + col];
#pragma unroll
        for (int r = 0; r < NRHS; ++r) {
            a0[r] = fma(l0, x[r * Nr + j0 + i], a0[r]);
            a1[r] = fma(l1, x[r * Nr + j0 + i + 1], a1[r]);
        }
    }
    if (rows & 1) {
        const double l0 = S[(long long)(j0 + rows - 1) * ld + col];
#pragma unroll
        for (int r = 0; r < NRHS; ++r) a0[r] = fma(l0, x[r * Nr + j0 + rows - 1], a0[r]);
    }
#pragma unroll
    for (int r = 0; r < NRHS; ++r) z[r * Nr + col] -= a0[r] + a1[r];
}

// Forward substitution L y = b in the same 32-block form, left-looking over the blocks b = 0 .. Nr/32-1 (the
// factorisation itself only forward-substitutes through its right-hand-side rows; chol_rcond.cu needs it for any
// vector).  Per block: the rows of b are reduced by L[rows of b, columns < 32 b] y (forward_reduce_block), then warp r
// solves the block's triangle for right-hand side r (solve_diag_block_lower, P from load_diag_block).

// One warp solves L_d y = r for the 32 entries r (lane k holds entry k) of one block; returns y the same way
__device__ __forceinline__ double solve_diag_block_lower(double r, const double* P, int lane) {
    const double rd = 1.0 / P[lane * LDQ + lane];
#pragma unroll
    for (int k = 0; k < NB; ++k) {
        const double yk = __shfl_sync(0xffffffffu, r * rd, k);
        if (lane == k) r = yk;
        if (lane > k) r = fma(-P[lane * LDQ + k], yk, r);
    }
    return r;
}

// z[r][row] -= sum_{j < j0} L[row][j] y[r][j] for the data rows row = j0 + i of block b (j0 = 32 b), i = warp, warp +
// NWARPS, ...: the lanes stride along the row (coalesced), then one warp sum per row.  z and y are [NRHS][Nr] and may be
// the same array.
template <int NRHS, int NWARPS>
__device__ __forceinline__ void forward_reduce_block(double* z, const double* y, const double* S, int ld, int Nr, int N,
                                                     int b, int warp, int lane) {
    constexpr int RPW = NB / NWARPS;
    const int j0 = NB * b;
    double acc[RPW][NRHS];
#pragma unroll
    for (int q = 0; q < RPW; ++q)
#pragma unroll
        for (int r = 0; r < NRHS; ++r) acc[q][r] = 0.0;
    for (int j = lane; j < j0; j += 32) {
        double yv[NRHS];
#pragma unroll
        for (int r = 0; r < NRHS; ++r) yv[r] = y[r * Nr + j];
#pragma unroll
        for (int q = 0; q < RPW; ++q) {
            const int row = j0 + warp + NWARPS * q;
            if (row < N) {
                const double l = S[(long long)row * ld + j];
#pragma unroll
                for (int r = 0; r < NRHS; ++r) acc[q][r] = fma(l, yv[r], acc[q][r]);
            }
        }
    }
#pragma unroll
    for (int q = 0; q < RPW; ++q) {
        const int row = j0 + warp + NWARPS * q;
#pragma unroll
        for (int r = 0; r < NRHS; ++r) {
            const double s = warp_sum(acc[q][r]);
            if (lane == 0 && row < N) z[r * Nr + row] -= s;
        }
    }
}

// Posterior scalars and weights of window w from the solution x[NRHS][Nr], v1 and the window's pivot status
// (read by thread 0 only).
// NRHS = 1: the conjugate (nu = (n1 + N + 2) w1 / (n1 - v1), :572-575) or Jeffreys (nu = w1, :600-606) weights;
// NRHS = 2: Jorion's Bayes-Stein estimator (:851-895) from y = C^-1 t and z = C^-1 1, see jorion_math.cuh.
// weights = (1/gamma) nu (:836, :849).
template <int NRHS, int NTHREADS>
__device__ __forceinline__ void write_outputs(const SolveParams& p, int w, const double* x, int Nr, double v1, int status,
                                              double* scratch) {
    const int tid = threadIdx.x;
    const int N = p.n_assets;
    const double* rhs = p.rhs + (long long)w * p.ldv;
    double* scal = p.scal + (long long)w * BP_S_COUNT;
    if constexpr (NRHS == 2) {
        const double* y = x;
        const double* z = x + Nr;
        double sy = 0.0, sz = 0.0, ty = 0.0;
        for (int j = tid; j < N; j += NTHREADS) {
            sy += y[j];
            sz += z[j];
            ty = fma(rhs[j], y[j], ty);
        }
        sy = block_sum(sy, scratch);
        sz = block_sum(sz, scratch);
        ty = block_sum(ty, scratch);
        const JorionCoef jc = jorion_coefficients(sy, sz, ty, (double)p.n_returns, (double)N);
        for (int j = tid; j < p.ldv; j += NTHREADS) {
            double yj = 0.0, nu = 0.0;
            if (j < N) {
                yj = y[j];
                nu = jc.c_y * yj + jc.c_z * z[j];
            }
            p.w1[(long long)w * p.ldv + j] = yj;
            p.nu[(long long)w * p.ldv + j] = nu;
            p.weights[(long long)w * p.ldv + j] = p.inv_gamma * nu;
        }
        if (tid == 0) {
            scal[BP_S_JORION_MU_G] = jc.mu_g;
            scal[BP_S_JORION_LAMBDA] = jc.lambda;
            scal[BP_S_JORION_V] = jc.v;
            scal[BP_S_JORION_Q] = jc.q;
            scal[BP_S_JORION_ONE_VINV_ONE] = jc.one_vinv_one;
        }
    } else {
        double mult = 1.0;
        if (p.mode == BP_MODE_CONJUGATE) {
            const double n1 = scal[BP_S_N1];
            mult = (n1 + (double)N + 2.0) / (n1 - v1);
        }
        for (int j = tid; j < p.ldv; j += NTHREADS) {
            const double wv = j < N ? x[j] : 0.0;
            const double nu = p.mode == BP_MODE_CONJUGATE ? (wv * mult) : wv;
            p.w1[(long long)w * p.ldv + j] = wv;
            p.nu[(long long)w * p.ldv + j] = nu;
            p.weights[(long long)w * p.ldv + j] = p.inv_gamma * nu;
        }
    }
    if (tid == 0) {
        scal[BP_S_V1] = v1;
        p.status[w] = status;
    }
}

}  // namespace chol
}  // namespace bp
