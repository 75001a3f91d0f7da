// Batched blocked Cholesky factorisation + triangular solves + posterior scalars.
//
// Replaces, per window, the reference's explicit inverse and mat-vec
//   w1 = inv(S1) (c S0 w0 + t)                      portfolio_calculations.py:485-489
//   nu = (n1 + N + 2) w1 / (n1 - w1' S1 w1)         :572-575      weights = (1/gamma) nu   :836
//   nu_J = inv(T - t t'/n) t                        :600-606      weights = (1/gamma) nu_J :849
// by S = L L', L z = b, L' w = z (SURVEY F8: within 1.5e-12 of inv()*b on well-posed inputs) and
// v1 = w1' S1 w1 = z'z.
//
// One CTA (4 warps) per window, 6 CTAs per SM (measured with the first TMA version: 4 -> 29.7 ms, 6 -> 26.4 ms,
// 8 -> 26.5 ms per step), left-looking blocked factorisation with 32-column panels, in place in the [rows][ldS] device layout produced by the Gram kernel (lower triangle):
//   U  panel update   C = S[j0:, j0:j0+32] - L[j0:, :j0] L[j0:j0+32, :j0]'   on the FP64 tensor cores.
//                     The already factored columns are streamed through shared memory by TMA
//                     (2-D tensor map over the whole workspace, 32-row x 16-column boxes,
//                     SWIZZLE_128B, 3-stage mbarrier ring) in slabs of 8*TPW m-tiles; each warp owns TPW
//                     8-row m-tiles of the slab and all four 8-column n-tiles of the panel.
//   F  diagonal block 32x32, blocked by 8 in FRAGMENT space: after the first slab the four warps that own its
//                     row blocks hold it in their accumulators; the warp owning a diagonal 8x8 tile computes its
//                     Cholesky factor and inverse in registers (warp shuffles, potrf8_inv8), the warps below
//                     solve / update their tiles with 2 DMMAs each.  (A single warp in shared memory was 2/3 of
//                     the kernel, CTA-wide 32-step loops in shared memory still 1/4.)
//   T  panel solve    L[j0+32:, j0:j0+32] = C * inv(L_d)' on the tensor cores, FUSED into the epilogue of
//                     the panel update: the accumulator fragment of a DMMA is, column for column, a valid
//                     A fragment (lane (g,tig) holds columns 8nt+2tig+h, which become the k slots of step
//                     (nt,h)), so C never goes to memory: the accumulators start as -S, collect +L L',
//                     go through a block forward substitution against L_d (8x8 inverses on the diagonal)
//                     in registers, and the finished factor rows are stored once.  (The first version wrote C and re-read it in a separate T phase: 2 MB of DRAM
//                     traffic per window and 15% of the kernel.)
// The factor is written with generic stores and re-read by TMA in later panels, so every panel ends
// with fence.proxy.async + a block barrier.  The right-hand side rides along as one extra row
// (row R = chol_rhs_row(N), kernels.h) of the matrix, so the forward substitution L z = b is a by-product
// of the factorisation.  R is the first 8-row tile after the data: for N mod 32 in 1..24 it lies in the
// padding rows below Nr = roundup(N,32), so the panels stop at row Nr - 1 instead of paying a whole slab
// (every chunk of the factored columns through the TMA ring) for one m-tile at row Nr; in the last panel
// the right-hand-side row then sits in the diagonal block, where it is solved by F and keeps an
// identity entry in its own padding column.  The back substitution then walks the panels in reverse
// with coalesced row reads and a warp-level triangular solve.
//
// k-permutation: inside a 16-column chunk, DMMA step q contracts columns {2q, 2q+1, 8+2q, 9+2q}
// over the four tig lanes.  With the 128-byte swizzle (16-byte unit index XOR row&7) the 16 lanes of
// a half warp then hit 16 distinct 8-byte words of the 128-byte bank line: every LDS.64 fragment
// load is conflict free.  A and B fragments use the same assignment, so the contraction is exact.
#include <cstdio>
#include <cstdlib>

#include "common.cuh"
#include "jorion_math.cuh"
#include "kernels.h"

namespace bp {

constexpr int NB = 32;

#ifndef CH_NWARPS
#define CH_NWARPS 4
#endif
constexpr int CH_WARPS = CH_NWARPS;                 // warps per window (CTA)
#ifndef CH_CTAS_PER_SM
#define CH_CTAS_PER_SM 6
#endif
constexpr int CH_OCC = CH_CTAS_PER_SM;              // resident CTAs (windows) per SM
constexpr int CH_THREADS = CH_WARPS * 32;

constexpr int LDQ = 34;    // row stride of the packed diagonal-block array

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

#ifndef CH_TPW
#define CH_TPW 2                                     // m-tiles per warp and slab
#endif
#ifndef CH_NSTAGES
#define CH_NSTAGES 2
#endif
constexpr int TPW = CH_TPW;
constexpr int SLAB_TILES = CH_WARPS * TPW;           // m-tiles per slab (one pass of the panel update)
constexpr int ABOXES = SLAB_TILES / 4;               // 32-row TMA boxes per slab
constexpr int CH_STAGES = CH_NSTAGES;
constexpr int BOX_BYTES = 32 * 16 * 8;               // one TMA box: 32 rows x 16 columns of doubles
constexpr int CH_STAGE_BYTES = (ABOXES + 1) * BOX_BYTES;   // A slab + 1 B box
constexpr int CH_TMA_SMEM = CH_STAGES * CH_STAGE_BYTES + 1024;

__device__ __forceinline__ void tma_load_2d(void* smem_dst, const void* tmap, int c0, int c1, uint64_t* bar) {
    asm volatile(
        "cp.async.bulk.tensor.2d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];"
        ::"r"(smem_u32(smem_dst)), "l"(reinterpret_cast<uint64_t>(tmap)), "r"(c0), "r"(c1), "r"(smem_u32(bar))
        : "memory");
}
// generic-proxy global writes (the factor) must be visible to later async-proxy (TMA) reads
__device__ __forceinline__ void fence_proxy_async_all() { asm volatile("fence.proxy.async.global;" ::: "memory"); }

// NRHS = 1: the posterior solves of the conjugate / Jeffreys path.  NRHS = 2 (Jorion, :851-895): a second
// right-hand side (the vector of ones) rides along as row R+1, so that both C^-1 t and C^-1 1 come out of ONE
// factorisation; the Bayes-Stein combination is the epilogue of this kernel.
template <int NRHS>
__global__ void __launch_bounds__(CH_THREADS, NRHS == 1 ? CH_OCC : 4)
chol_solve_kernel(const __grid_constant__ CUtensorMap smap, const SolveParams p) {
    extern __shared__ unsigned char sm_raw[];
    __shared__ uint64_t full_bar[CH_STAGES];
    __shared__ uint64_t empty_bar[CH_STAGES];     // one arrival per consumer warp
    __shared__ int fail_s;
    // 1024-byte alignment by pointer arithmetic on the shared array (keeps the shared address space)
    unsigned char* stage_mem = sm_raw + ((1024u - (smem_u32(sm_raw) & 1023u)) & 1023u);
    double* P = reinterpret_cast<double*>(stage_mem + CH_STAGES * CH_STAGE_BYTES);   // [32][LDQ]: L_d (lower) + inv(L_d)' (upper)
    double* scratch = P + NB * LDQ;        // [40]
    // solution vectors of the back substitution: alias the TMA stages (after the last panel they are idle)
    double* xs = reinterpret_cast<double*>(stage_mem);   // [NRHS][Nr]

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int g = lane >> 2, tig = lane & 3;
    const int N = p.n_assets;
    const int ld = p.ldS;
    const int Nr = (N + NB - 1) / NB * NB;
    const int R = chol_rhs_row(N);             // row index of the right-hand side
    const int rows_end = max(Nr, R + 8);       // the panels cover rows j0 .. rows_end-1
    const int rowsS = (int)(p.win_stride / ld);

    if (tid == 0) {
        tma_prefetch_desc(&smap);
        for (int s = 0; s < CH_STAGES; ++s) {
            mbar_init(&full_bar[s], 1);
            mbar_init(&empty_bar[s], CH_WARPS);
        }
        fence_barrier_init();
        fence_proxy_async();
    }
    __syncthreads();
    // per-lane fragment offsets inside a [32][16] swizzled box: row r = 8*t + g, DMMA step q reads column
    // c = 2q + (tig&1) + 8*(tig>>1): 16-byte unit (q + 4*(tig>>1)) ^ g, 8-byte half tig&1
    int foff[4];
#pragma unroll
    for (int q = 0; q < 4; ++q) foff[q] = g * 128 + (((q + 4 * (tig >> 1)) ^ g) << 4) + (tig & 1) * 8;
    uint32_t it = 0;      // chunks consumed so far (mbarrier phase bookkeeping)
    // optional phase profile (BP_CHOL_PROFILE=1): cycles of thread 0 between phase boundaries
    long long prof[6] = {0, 0, 0, 0, 0, 0};
    long long tlast = p.debug ? clock64() : 0;
#define PROF(k)                                   \
    if (p.debug && tid == 0) {                    \
        const long long tn = clock64();           \
        prof[k] += tn - tlast;                    \
        tlast = tn;                               \
    }

    // CTA job q factorises window q * w_stride: the loop runs over the window index itself
    for (int w = blockIdx.x * max(p.w_stride, 1); w < p.n_windows * max(p.w_stride, 1); w += gridDim.x * max(p.w_stride, 1)) {
        double* S = p.S + (long long)w * p.win_stride;
        const double* rhs = p.rhs + (long long)w * p.ldv;
        const int grow0 = w * rowsS;           // first row of this window in the tensor map
        if (tid == 0) fail_s = 0;
        for (int j = tid; j < ld; j += CH_THREADS) S[(long long)R * ld + j] = j < N ? rhs[j] : 0.0;
        if constexpr (NRHS == 2)
            for (int j = tid; j < ld; j += CH_THREADS) S[(long long)(R + 1) * ld + j] = j < N ? 1.0 : 0.0;
        fence_proxy_async_all();
        __syncthreads();

        for (int j0 = 0; j0 < N; j0 += NB) {
            const int mt_total = (rows_end - j0) / 8;      // m-tiles covering rows j0 .. rows_end-1
            const int nchunks = j0 / 16;
            // ---------------- U (+F after the first slab) + fused T, one slab of SLAB_TILES m-tiles per pass
            for (int slab0 = 0; slab0 < mt_total; slab0 += SLAB_TILES) {
                const int slab_tiles = min(SLAB_TILES, mt_total - slab0);
                const int nboxes = (slab_tiles + 3) >> 2;
                const int slab_row = j0 + 8 * slab0;
                int ni = 0;                  // m-tiles this warp really has in this slab (warp-uniform)
#pragma unroll
                for (int i = 0; i < TPW; ++i) ni += (warp + CH_WARPS * i) < slab_tiles ? 1 : 0;

                auto issue = [&](int c, uint32_t seq) {
                    const int stage = seq % CH_STAGES;
                    unsigned char* dst = stage_mem + stage * CH_STAGE_BYTES;
                    // the stage is free once all consumer warps have released its previous use
                    if (seq >= CH_STAGES) mbar_wait(&empty_bar[stage], ((seq / CH_STAGES) - 1) & 1);
                    mbar_arrive_expect_tx(&full_bar[stage], (uint32_t)(nboxes + 1) * BOX_BYTES);
                    for (int bx = 0; bx < nboxes; ++bx)
                        tma_load_2d(dst + bx * BOX_BYTES, &smap, 16 * c, grow0 + slab_row + 32 * bx, &full_bar[stage]);
                    tma_load_2d(dst + ABOXES * BOX_BYTES, &smap, 16 * c, grow0 + j0, &full_bar[stage]);
                };
                if (tid == 0)
                    for (int c = 0; c < CH_STAGES && c < nchunks; ++c) issue(c, it + c);

                // accumulators start as -S (identity rows for the padding), collect +L L': acc = -C
                double acc[TPW][4][2];
#pragma unroll
                for (int i = 0; i < TPW; ++i) {
                    const int row = j0 + 8 * (slab0 + warp + CH_WARPS * i) + g;
                    const bool real = i < ni && (row < N || (row >= R && row < R + NRHS));
#pragma unroll
                    for (int nt = 0; nt < 4; ++nt) {
                        const int col = j0 + 8 * nt + 2 * tig;
                        double2 sv = make_double2(0.0, 0.0);
                        if (real && col < N) sv = *reinterpret_cast<const double2*>(S + (long long)row * ld + col);
                        if (real) {
                            acc[i][nt][0] = -sv.x;
                            acc[i][nt][1] = col + 1 < N ? -sv.y : 0.0;
                        } else {
                            acc[i][nt][0] = row == col ? -1.0 : 0.0;
                            acc[i][nt][1] = row == col + 1 ? -1.0 : 0.0;
                        }
                    }
                }

                for (int c = 0; c < nchunks; ++c, ++it) {
                    const int stage = it % CH_STAGES;
                    const unsigned char* sA = stage_mem + stage * CH_STAGE_BYTES;
                    const unsigned char* sB = sA + ABOXES * BOX_BYTES;
                    mbar_wait(&full_bar[stage], (it / CH_STAGES) & 1);
                    if (ni == TPW) {
                        // full slab (all but the last slab of a panel): no per-tile predicate, so the loads of a k-step
                        // are issued together and its TPW x 4 DMMAs follow without branches or re-convergence points
#pragma unroll
                        for (int q = 0; q < 4; ++q) {
                            double b[4], a[TPW];
#pragma unroll
                            for (int nt = 0; nt < 4; ++nt)
                                b[nt] = *reinterpret_cast<const double*>(sB + nt * 1024 + foff[q]);
#pragma unroll
                            for (int i = 0; i < TPW; ++i) {
                                const int t = warp + CH_WARPS * i;
                                a[i] = *reinterpret_cast<const double*>(sA + (t >> 2) * BOX_BYTES + (t & 3) * 1024 + foff[q]);
                            }
#pragma unroll
                            for (int i = 0; i < TPW; ++i)
#pragma unroll
                                for (int nt = 0; nt < 4; ++nt) dmma884(acc[i][nt][0], acc[i][nt][1], a[i], b[nt]);
                        }
                    } else {
#pragma unroll
                    for (int q = 0; q < 4; ++q) {
                        double b[4];
#pragma unroll
                        for (int nt = 0; nt < 4; ++nt)
                            b[nt] = *reinterpret_cast<const double*>(sB + nt * 1024 + foff[q]);
#pragma unroll
                        for (int i = 0; i < TPW; ++i) {
                            if (i < ni) {    // skip the m-tile slots past the end of the slab
                                const int t = warp + CH_WARPS * i;
                                const double a = *reinterpret_cast<const double*>(sA + (t >> 2) * BOX_BYTES + (t & 3) * 1024 + foff[q]);
#pragma unroll
                                for (int nt = 0; nt < 4; ++nt) dmma884(acc[i][nt][0], acc[i][nt][1], a, b[nt]);
                            }
                        }
                    }
                    }
                    __syncwarp();
                    if (lane == 0) mbar_arrive(&empty_bar[stage]);   // this warp is done with the stage
                    if (tid == 0 && c + CH_STAGES < nchunks) issue(c + CH_STAGES, it + CH_STAGES);
                }

                // padding: rows N..rows_end-1 other than the right-hand sides, and columns >= N, hold no data;
                // whatever the update accumulated there is replaced by the identity.  In a padding column that is
                // zero for the rows of S and a unit diagonal for a right-hand-side row R < Nr, which sits in the
                // diagonal block of the last panel: its pivot must not be zero
                if (slab_row + 8 * slab_tiles > N || j0 + NB > N) {
#pragma unroll
                    for (int i = 0; i < TPW; ++i) {
                        const int row = j0 + 8 * (slab0 + warp + CH_WARPS * i) + g;
                        const bool real = row < N || (row >= R && row < R + NRHS);
#pragma unroll
                        for (int nt = 0; nt < 4; ++nt) {
                            const int col = j0 + 8 * nt + 2 * tig;
                            if (!real || col >= N) acc[i][nt][0] = row == col ? -1.0 : 0.0;
                            if (!real || col + 1 >= N) acc[i][nt][1] = row == col + 1 ? -1.0 : 0.0;
                        }
                    }
                }

                if (slab0 == 0) {
                    // ---------------- F: 32x32 diagonal block, blocked by 8 in fragment space.  Warp q < 4 holds
                    // row block q (acc[0][0..3] = -C).  Column block cb: warp cb factors and inverts its 8x8
                    // tile in registers; the warps below solve their tile against it (2 DMMAs) and update their
                    // remaining tiles (2 DMMAs each); L goes to the lower part of P, W' to the upper part.
                    PROF(0)
#pragma unroll
                    for (int cb = 0; cb < NB / 8; ++cb) {
                        if (warp == cb) {
                            double d0 = -acc[0][cb][0], d1 = -acc[0][cb][1], y0, y1;
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
                            for (int h = 0; h < 2; ++h) dmma884(x0, x1, acc[0][cb][h], wfrag(P, cb, cb, h, g, tig));
                            x0 = -x0;
                            x1 = -x1;
                            acc[0][cb][0] = x0;      // this tile now holds +L
                            acc[0][cb][1] = x1;
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
                                        dmma884(acc[0][nb][0], acc[0][nb][1], acc[0][cb][h], wfrag(P, cb, nb, h, g, tig));
                                }
                        }
                    }
                    PROF(1)
                    // write L_d back (lower part, real rows only: in the last panel z of a right-hand side R < Nr)
                    for (int i = warp; i < NB; i += CH_WARPS) {
                        const int row = j0 + i, col = j0 + lane;
                        if ((row < N || (row >= R && row < R + NRHS)) && col < N && lane <= i)
                            S[(long long)row * ld + col] = P[i * LDQ + lane];
                    }
                }
                // ---------------- T: X = C inv(L_d)' straight from the accumulators, by block forward substitution
                // with W: X_cb = C_cb inv(L_cb,cb)', C_nb -= X_cb L_nb,cb' (nb > cb).  DMMA step h contracts the
                // columns 8cb+2tig+h the lanes already hold, so the accumulators are used as A fragments as they are.
#pragma unroll
                for (int i = 0; i < TPW; ++i) {
                    const int q = slab0 + warp + CH_WARPS * i;     // m-tile index within the panel
                    if (i >= ni || q < NB / 8) continue;
                    const int row = j0 + 8 * q + g;
                    const bool real = row < N || (row >= R && row < R + NRHS);
#pragma unroll
                    for (int cb = 0; cb < NB / 8; ++cb) {
                        double x0 = 0.0, x1 = 0.0;
#pragma unroll
                        for (int h = 0; h < 2; ++h) dmma884(x0, x1, acc[i][cb][h], wfrag(P, cb, cb, h, g, tig));
                        x0 = -x0;
                        x1 = -x1;
                        const int col = j0 + 8 * cb + 2 * tig;
                        if (real && col < N) *reinterpret_cast<double2*>(S + (long long)row * ld + col) = make_double2(x0, x1);
#pragma unroll
                        for (int nb = cb + 1; nb < NB / 8; ++nb) {
                            dmma884(acc[i][nb][0], acc[i][nb][1], x0, wfrag(P, cb, nb, 0, g, tig));
                            dmma884(acc[i][nb][0], acc[i][nb][1], x1, wfrag(P, cb, nb, 1, g, tig));
                        }
                    }
                }
            }
            fence_proxy_async_all();        // the factor written above is read by TMA in the next panels
            __syncthreads();
            PROF(2)
        }

        // ---------------- z = L^-1 b sits in row R (+r);  v1 = z'z = w1' S1 w1   (:574)
        double zz = 0.0;
        for (int j = tid; j < Nr; j += CH_THREADS) {
            const double z = j < N ? S[(long long)R * ld + j] : 0.0;
            xs[j] = z;
            zz = fma(z, z, zz);
            if constexpr (NRHS == 2) xs[Nr + j] = j < N ? S[(long long)(R + 1) * ld + j] : 0.0;
        }
        const double v1 = block_sum(zz, scratch);

        // ---------------- back substitution  L' x = z, right-looking over 32-column blocks, in place in xs: block b is
        // solved (warp r finishes right-hand side r), then every block bb < b is reduced by L[rows of b, columns of bb]' x_b
        // (one warp per block, coalesced rows).  Operation for operation the arithmetic of chol_cluster.cu, so that a
        // batch gives bit-identical weights however its windows are split over launches and kernels.
        for (int b = Nr / NB - 1; b >= 0; --b) {
            const int j0 = NB * b;
            for (int i = warp; i < NB; i += CH_WARPS) {
                const int row = j0 + i, col = j0 + lane;
                double v;
                if (row < N && col < N) v = lane <= i ? S[(long long)row * ld + col] : 0.0;
                else v = i == lane ? 1.0 : 0.0;
                P[i * LDQ + lane] = v;
            }
            __syncthreads();
            if (warp < NRHS) {
                double r = xs[warp * Nr + j0 + lane];
                const double rd = 1.0 / P[lane * LDQ + lane];      // all 32 reciprocals in parallel
#pragma unroll
                for (int k = NB - 1; k >= 0; --k) {
                    const double xk = __shfl_sync(0xffffffffu, r * rd, k);
                    if (lane == k) r = xk;
                    if (lane < k) r = fma(-P[k * LDQ + lane], xk, r);
                }
                xs[warp * Nr + j0 + lane] = r;
            }
            __syncthreads();
            const int rows = min(NB, N - j0);
            for (int bb = warp; bb < b; bb += CH_WARPS) {
                const int col = NB * bb + lane;
                double a0[NRHS], a1[NRHS];
#pragma unroll
                for (int r = 0; r < NRHS; ++r) a0[r] = a1[r] = 0.0;
#pragma unroll 4
                for (int i = 0; i + 1 < rows; i += 2) {
                    const double l0 = S[(long long)(j0 + i) * ld + col], l1 = S[(long long)(j0 + i + 1) * ld + col];
#pragma unroll
                    for (int r = 0; r < NRHS; ++r) {
                        a0[r] = fma(l0, xs[r * Nr + j0 + i], a0[r]);
                        a1[r] = fma(l1, xs[r * Nr + j0 + i + 1], a1[r]);
                    }
                }
                if (rows & 1) {
                    const double l0 = S[(long long)(j0 + rows - 1) * ld + col];
#pragma unroll
                    for (int r = 0; r < NRHS; ++r) a0[r] = fma(l0, xs[r * Nr + j0 + rows - 1], a0[r]);
                }
#pragma unroll
                for (int r = 0; r < NRHS; ++r) xs[r * Nr + col] -= a0[r] + a1[r];
            }
        }
        __syncthreads();

        PROF(3)
        // ---------------- posterior scalars and weights
        double* scal = p.scal + (long long)w * BP_S_COUNT;
        if constexpr (NRHS == 2) {
            // Jorion's Bayes-Stein estimator (:851-895) from y = C^-1 t and z = C^-1 1: see jorion_math.cuh
            const double* y = xs;
            const double* z = xs + Nr;
            double sy = 0.0, sz = 0.0, ty = 0.0;
            for (int j = tid; j < N; j += CH_THREADS) {
                sy += y[j];
                sz += z[j];
                ty = fma(rhs[j], y[j], ty);
            }
            sy = block_sum(sy, scratch);
            sz = block_sum(sz, scratch);
            ty = block_sum(ty, scratch);
            const JorionCoef jc = jorion_coefficients(sy, sz, ty, (double)p.n_returns, (double)N);
            for (int j = tid; j < p.ldv; j += CH_THREADS) {
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
        for (int j = tid; j < p.ldv; j += CH_THREADS) {
            const double wv = j < N ? xs[j] : 0.0;
            const double nu = p.mode == BP_MODE_CONJUGATE ? (wv * mult) : wv;
            p.w1[(long long)w * p.ldv + j] = wv;
            p.nu[(long long)w * p.ldv + j] = nu;
            p.weights[(long long)w * p.ldv + j] = p.inv_gamma * nu;
        }
        }
        if (tid == 0) {
            scal[BP_S_V1] = v1;
            p.status[w] = fail_s;
        }
        __syncthreads();
        PROF(4)
    }
    if (p.debug && tid == 0)
        for (int k = 0; k < 6; ++k) atomicAdd(reinterpret_cast<unsigned long long*>(p.debug) + k, (unsigned long long)prof[k]);
#undef PROF
}

// windows the solver works on concurrently (one CTA each): a launch of a multiple of this runs full waves
int chol_wave_windows(int sm_count) {
    static const int ctas_per_sm = [] {
        const char* e = getenv("BP_CHOL_CTAS_PER_SM");      // tuning knob (default: CH_OCC)
        const int v = e ? atoi(e) : CH_OCC;
        return v >= 1 && v <= CH_OCC ? v : CH_OCC;
    }();
    return ctas_per_sm * sm_count;
}

size_t chol_smem_bytes(int n_assets, int nrhs) {
    const int Nr = (n_assets + NB - 1) / NB * NB;
    // xs aliases the stage ring: it must hold it
    if ((size_t)CH_STAGES * CH_STAGE_BYTES < sizeof(double) * (size_t)Nr * nrhs) return 0;
    return (size_t)CH_TMA_SMEM + sizeof(double) * (size_t)(NB * LDQ + 40);
}

int chol_max_assets(int nrhs) {
    return (int)((size_t)CH_STAGES * CH_STAGE_BYTES / (sizeof(double) * (size_t)nrhs)) / NB * NB;
}

cudaError_t launch_chol_solve(const SolveParams& p, const CUtensorMap& smap, int sm_count, cudaStream_t st) {
    if (p.n_windows <= 0) return cudaSuccess;
    static const bool profile = getenv("BP_CHOL_PROFILE") != nullptr;
    if (!profile) {
        // launches too small to fill the machine: one thread-block cluster per window (chol_cluster.cu)
        const cudaError_t ec = launch_chol_cluster(p, smap, chol_wave_windows(sm_count), st);
        if (ec != cudaErrorNotSupported) return ec;
    }
    const int nrhs = p.estimator == BP_EST_JORION ? 2 : 1;
    const size_t smem = chol_smem_bytes(p.n_assets, nrhs);
    if (smem == 0) return cudaErrorInvalidValue;      // N too large for the aliased back-substitution vector
    cudaError_t e = nrhs == 2 ? cudaFuncSetAttribute(chol_solve_kernel<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)
                              : cudaFuncSetAttribute(chol_solve_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    int grid = chol_wave_windows(sm_count);
    if (grid > p.n_windows) grid = p.n_windows;
    if (nrhs == 2) {
        chol_solve_kernel<2><<<grid, CH_THREADS, smem, st>>>(smap, p);
        return cudaGetLastError();
    }
    if (profile) {
        SolveParams q = p;
        static long long* dbg = nullptr;
        if (!dbg) cudaMalloc(&dbg, 6 * sizeof(long long));
        cudaMemsetAsync(dbg, 0, 6 * sizeof(long long), st);
        q.debug = dbg;
        chol_solve_kernel<1><<<grid, CH_THREADS, smem, st>>>(smap, q);
        long long hostv[6];
        cudaMemcpyAsync(hostv, dbg, sizeof(hostv), cudaMemcpyDeviceToHost, st);
        cudaStreamSynchronize(st);
        const double tot = (double)(hostv[0] + hostv[1] + hostv[2] + hostv[3] + hostv[4]);
        fprintf(stderr, "[chol profile] W=%d U(slab0)=%.1f%% F=%.1f%% U+T(rest)=%.1f%% backsub=%.1f%% out=%.1f%% cycles/window=%.0f\n", p.n_windows,
                100 * hostv[0] / tot, 100 * hostv[1] / tot, 100 * hostv[2] / tot, 100 * hostv[3] / tot, 100 * hostv[4] / tot,
                tot / p.n_windows);
        return cudaGetLastError();
    }
    chol_solve_kernel<1><<<grid, CH_THREADS, smem, st>>>(smap, p);
    return cudaGetLastError();
}

}  // namespace bp
