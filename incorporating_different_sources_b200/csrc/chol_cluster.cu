// Batched blocked Cholesky + triangular solves + posterior scalars, ONE THREAD-BLOCK CLUSTER PER WINDOW.
//
// Same mathematics and the same panel kernels as chol_solve.cu (left-looking, 32-column panels, TMA-fed DMMA panel
// update with the panel solve fused into its epilogue, register-level 32x32 diagonal block; w1 = inv(S1)(c S0 w0 + t)
// :485-489, nu :572-575, Jeffreys :600-606, weights = (1/gamma) nu :836,:849), but the rows of a window are spread
// over the K CTAs of a cluster instead of one CTA doing everything.  The right-hand side(s) ride along as rows R, R+1
// of the factorisation with R = chol_rhs_row(N), exactly as there, so that both kernels give the same bits.
//
// Why: (1) latency -- a launch of a few windows (one façade call, the 65 Jeffreys base windows of a date-range shard on
// 8 GPUs) leaves most SMs idle with one 4-warp CTA per window; K CTAs per window finish it roughly K times sooner.
// (2) An experiment on the DRAM traffic of full launches: the left-looking update re-reads the factored columns once
// per panel (5.2 MB per window at N = 500); with 888 windows in flight the L2 holds a quarter of the hot factors
// (10.7 MB of DRAM reads per window, hit rate 27 %, HBM at 72 % of its peak).  148 windows in flight bring that down
// to 2.96 MB (profiles/r2_solver_l2_probe.txt), and clusters of 4 halve the traffic (5.4 MB) -- but the serial parts
// of a factorisation (diagonal blocks, the back-substitution chain) idle the other CTAs of the cluster and at N = 500
// there are too few 32-row groups per panel to hide them (cluster-barrier waits = 35 % of the stall samples), so the
// full launches stay with chol_solve_kernel (see chol_cluster_size below for the measured times).
//
// Work split inside a cluster (rank r of K), panel p (columns j0 = 32 p):
//   * the rows below the panel are cut into GROUPS of 32 rows (one TMA box, one 8-row m-tile per warp); group q
//     belongs to CTA (q + p) mod K, so that the diagonal group (q = 0) rotates over the CTAs; a CTA takes its groups
//     two at a time (one pass = 2 A boxes + 1 B box per 16-column chunk, exactly the slab of chol_solve.cu);
//   * the owner of the diagonal group factors the 32x32 block in registers after its first pass and PUSHES the packed
//     block (L_d below, inv-diagonal-tiles transposed above: 8.7 KB) into the shared memory of its peers (DSMEM
//     stores), then arrives on the cluster barrier; the peers arrive BEFORE their first pass and wait after it, so the
//     diagonal block is hidden behind their panel update;
//   * the finished factor rows go to global memory with generic stores and are re-read by the TMA of EVERY CTA in the
//     next panel: fence.proxy.async + cluster barrier (release / acquire) at the end of each panel.
// Back substitution L'x = z, right-looking over column blocks: CTA b mod K owns the 32 unknowns of block b and the
// running right-hand side of its blocks; per block the owner solves the 32x32 triangle (warp shuffles), pushes x_b to
// every CTA, one cluster barrier, then every CTA subtracts L[b rows, its blocks] x_b from its own blocks (one warp per
// block, coalesced rows).  One cluster barrier per block instead of a cross-CTA reduction.
#include <cooperative_groups.h>
#include <cstdio>
#include <cstdlib>

#include "common.cuh"
#include "jorion_math.cuh"
#include "kernels.h"

namespace cg = cooperative_groups;

namespace bp {

namespace {

constexpr int NB = 32;
constexpr int CC_WARPS = 4;
constexpr int CC_THREADS = CC_WARPS * 32;
#ifndef CC_CTAS_PER_SM
#define CC_CTAS_PER_SM 6
#endif
constexpr int CC_OCC = CC_CTAS_PER_SM;
constexpr int LDQ = 34;                              // row stride of the packed diagonal-block array
constexpr int TPW = 2;                               // groups (A boxes) per pass = m-tiles per warp and pass
constexpr int CC_STAGES = 2;
constexpr int BOX_BYTES = 32 * 16 * 8;               // one TMA box: 32 rows x 16 columns of doubles
constexpr int CC_STAGE_BYTES = (TPW + 1) * BOX_BYTES;   // A boxes + 1 B box
constexpr int CC_TMA_SMEM = CC_STAGES * CC_STAGE_BYTES + 1024;
constexpr int CC_MAX_CLUSTER = 8;

// Cholesky factor AND inverse of one 8x8 diagonal tile by one warp in registers (see chol_solve.cu: potrf8_inv8).
// The tile is in DMMA accumulator layout; on return d0/d1 hold L, y0/y1 inv(L).  Returns the 1-based index of the
// first non-positive pivot, or 0.
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

// B fragment of the panel solve from the packed block P (L below the diagonal, W' = L with inverted diagonal tiles,
// transposed and shifted by one column, above it); conflict free, see chol_solve.cu
__device__ __forceinline__ double wfrag(const double* P, int kb, int nb, int h, int g, int tig) {
    const double v = P[(8 * kb + 2 * tig + h) * LDQ + 8 * nb + g + 1];
    return (nb == kb && 2 * tig + h > g) ? 0.0 : v;
}

__device__ __forceinline__ void tma_load_2d(void* smem_dst, const void* tmap, int c0, int c1, uint64_t* bar) {
    asm volatile(
        "cp.async.bulk.tensor.2d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];"
        ::"r"(smem_u32(smem_dst)), "l"(reinterpret_cast<uint64_t>(tmap)), "r"(c0), "r"(c1), "r"(smem_u32(bar))
        : "memory");
}
// generic-proxy global writes (the factor) must be visible to later async-proxy (TMA) reads, here and in the peers
__device__ __forceinline__ void fence_proxy_async_all() { asm volatile("fence.proxy.async.global;" ::: "memory"); }
__device__ __forceinline__ void cluster_arrive() { asm volatile("barrier.cluster.arrive.release;" ::: "memory"); }
__device__ __forceinline__ void cluster_wait() { asm volatile("barrier.cluster.wait.acquire;" ::: "memory"); }

}  // namespace

template <int NRHS>
__global__ void __launch_bounds__(CC_THREADS, CC_OCC)
chol_cluster_kernel(const __grid_constant__ CUtensorMap smap, const SolveParams p) {
    extern __shared__ unsigned char sm_raw[];
    __shared__ uint64_t full_bar[CC_STAGES];
    __shared__ uint64_t empty_bar[CC_STAGES];     // one arrival per consumer warp
    __shared__ int fail_s;
    __shared__ int fail_all[CC_MAX_CLUSTER];      // rank 0: first failing column reported by every CTA
    unsigned char* stage_mem = sm_raw + ((1024u - (smem_u32(sm_raw) & 1023u)) & 1023u);
    double* P = reinterpret_cast<double*>(stage_mem + CC_STAGES * CC_STAGE_BYTES);   // [32][LDQ]
    double* scratch = P + NB * LDQ;               // [40]

    cg::cluster_group cluster = cg::this_cluster();
    const int K = (int)cluster.num_blocks();
    const int rank = (int)cluster.block_rank();
    const int cid = blockIdx.x / K, ncl = gridDim.x / K;

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int g = lane >> 2, tig = lane & 3;
    const int N = p.n_assets;
    const int ld = p.ldS;
    const int Nr = (N + NB - 1) / NB * NB;
    const int R = chol_rhs_row(N);             // row index of the right-hand side (see chol_solve.cu)
    const int rows_end = max(Nr, R + 8);       // the panels cover rows j0 .. rows_end-1
    const int rowsS = (int)(p.win_stride / ld);
    const int stride = max(p.w_stride, 1);
    // back substitution vectors alias the TMA stages (idle after the last panel): running rhs and solution
    double* zs = reinterpret_cast<double*>(stage_mem);   // [NRHS][Nr]
    double* xsol = zs + NRHS * Nr;                        // [NRHS][Nr]

    if (tid == 0) {
        tma_prefetch_desc(&smap);
        for (int s = 0; s < CC_STAGES; ++s) {
            mbar_init(&full_bar[s], 1);
            mbar_init(&empty_bar[s], CC_WARPS);
        }
        fence_barrier_init();
        fence_proxy_async();
    }
    __syncthreads();
    int foff[4];
#pragma unroll
    for (int q = 0; q < 4; ++q) foff[q] = g * 128 + (((q + 4 * (tig >> 1)) ^ g) << 4) + (tig & 1) * 8;
    uint32_t it = 0;      // chunks consumed so far (mbarrier phase bookkeeping)

    for (int wq = cid; wq < p.n_windows; wq += ncl) {
        const int w = wq * stride;
        double* S = p.S + (long long)w * p.win_stride;
        const double* rhs = p.rhs + (long long)w * p.ldv;
        const int grow0 = w * rowsS;           // first row of this window in the tensor map
        if (tid == 0) fail_s = 0;
        __syncthreads();

        for (int j0 = 0, pi = 0; j0 < N; j0 += NB, ++pi) {
            const int mt_total = (rows_end - j0) / 8;      // m-tiles covering rows j0 .. rows_end-1
            const int ng = (mt_total + 3) >> 2;            // 32-row groups
            const int nchunks = j0 / 16;
            const bool diag_owner = rank == pi % K;
            const int qfirst = ((rank - pi) % K + K) % K;
            if (!diag_owner) cluster_arrive();             // barrier A ("diagonal block pushed"), arrive early
            bool waitedA = false;

            for (int q0 = qfirst; q0 < ng; q0 += TPW * K) {
                const int nboxes = (q0 + K < ng) ? 2 : 1;
                int ni = 0;                  // m-tiles this warp really has in this pass (warp-uniform)
#pragma unroll
                for (int i = 0; i < TPW; ++i) ni += (q0 + i * K < ng && 4 * (q0 + i * K) + warp < mt_total) ? 1 : 0;

                auto issue = [&](int c, uint32_t seq) {
                    const int stage = seq % CC_STAGES;
                    unsigned char* dst = stage_mem + stage * CC_STAGE_BYTES;
                    if (seq >= CC_STAGES) mbar_wait(&empty_bar[stage], ((seq / CC_STAGES) - 1) & 1);
                    mbar_arrive_expect_tx(&full_bar[stage], (uint32_t)(nboxes + 1) * BOX_BYTES);
                    for (int bx = 0; bx < nboxes; ++bx)
                        tma_load_2d(dst + bx * BOX_BYTES, &smap, 16 * c, grow0 + j0 + 32 * (q0 + bx * K), &full_bar[stage]);
                    tma_load_2d(dst + TPW * BOX_BYTES, &smap, 16 * c, grow0 + j0, &full_bar[stage]);
                };
                if (tid == 0)
                    for (int c = 0; c < CC_STAGES && c < nchunks; ++c) issue(c, it + c);

                // accumulators start as -S (identity rows for the padding), collect +L L': acc = -C
                double acc[TPW][4][2];
#pragma unroll
                for (int i = 0; i < TPW; ++i) {
                    const int row = j0 + 32 * (q0 + i * K) + 8 * warp + g;
                    const bool real = i < ni && (row < N || (row >= R && row < R + NRHS));
#pragma unroll
                    for (int nt = 0; nt < 4; ++nt) {
                        const int col = j0 + 8 * nt + 2 * tig;
                        double2 sv = make_double2(0.0, 0.0);
                        if (real && col < N) {
                            if (row < N) sv = *reinterpret_cast<const double2*>(S + (long long)row * ld + col);
                            else if (NRHS == 2 && row == R + 1) sv = make_double2(1.0, 1.0);
                            else sv = *reinterpret_cast<const double2*>(rhs + col);     // the right-hand side rides along as row R
                        }
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
                    const int stage = it % CC_STAGES;
                    const unsigned char* sA = stage_mem + stage * CC_STAGE_BYTES;
                    const unsigned char* sB = sA + TPW * BOX_BYTES;
                    mbar_wait(&full_bar[stage], (it / CC_STAGES) & 1);
#pragma unroll
                    for (int q = 0; q < 4; ++q) {
                        double b[4];
#pragma unroll
                        for (int nt = 0; nt < 4; ++nt)
                            b[nt] = *reinterpret_cast<const double*>(sB + nt * 1024 + foff[q]);
#pragma unroll
                        for (int i = 0; i < TPW; ++i) {
                            if (i < ni) {
                                const double a = *reinterpret_cast<const double*>(sA + i * BOX_BYTES + warp * 1024 + foff[q]);
#pragma unroll
                                for (int nt = 0; nt < 4; ++nt) dmma884(acc[i][nt][0], acc[i][nt][1], a, b[nt]);
                            }
                        }
                    }
                    __syncwarp();
                    if (lane == 0) mbar_arrive(&empty_bar[stage]);   // this warp is done with the stage
                    if (tid == 0 && c + CC_STAGES < nchunks) issue(c + CC_STAGES, it + CC_STAGES);
                }

                // padding: rows N..rows_end-1 other than the right-hand sides, and columns >= N, hold no data;
                // whatever the update accumulated there is replaced by the identity (zero for the rows of S, a unit
                // diagonal for a right-hand-side row R < Nr in the diagonal block of the last panel)
                if (j0 + 32 * (q0 + (nboxes - 1) * K) + 32 > N || j0 + NB > N) {
#pragma unroll
                    for (int i = 0; i < TPW; ++i) {
                        const int row = j0 + 32 * (q0 + i * K) + 8 * warp + g;
                        const bool real = row < N || (row >= R && row < R + NRHS);
#pragma unroll
                        for (int nt = 0; nt < 4; ++nt) {
                            const int col = j0 + 8 * nt + 2 * tig;
                            if (!real || col >= N) acc[i][nt][0] = row == col ? -1.0 : 0.0;
                            if (!real || col + 1 >= N) acc[i][nt][1] = row == col + 1 ? -1.0 : 0.0;
                        }
                    }
                }

                if (q0 == 0) {
                    // ---------------- F: 32x32 diagonal block in fragment space (this CTA owns the diagonal group)
#pragma unroll
                    for (int cb = 0; cb < NB / 8; ++cb) {
                        if (warp == cb) {
                            double d0 = -acc[0][cb][0], d1 = -acc[0][cb][1], y0, y1;
                            const int f = potrf8_inv8(d0, d1, y0, y1, g, tig, lane);
                            // tiles from row N on: padding and right-hand sides, no pivots of S (see chol_solve.cu)
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
                    // push the packed block to the peers, then barrier A; write L_d back (lower part, real rows only:
                    // in the last panel z of a right-hand side R < Nr)
                    for (int peer = 0; peer < K; ++peer) {
                        if (peer == rank) continue;
                        double* dst = cluster.map_shared_rank(P, peer);
                        for (int e = tid; e < NB * LDQ; e += CC_THREADS) dst[e] = P[e];
                    }
                    cluster_arrive();
                    for (int i = warp; i < NB; i += CC_WARPS) {
                        const int row = j0 + i, col = j0 + lane;
                        if ((row < N || (row >= R && row < R + NRHS)) && col < N && lane <= i)
                            S[(long long)row * ld + col] = P[i * LDQ + lane];
                    }
                }
                if (!waitedA) {
                    cluster_wait();
                    waitedA = true;
                }
                // ---------------- T: X = C inv(L_d)' straight from the accumulators (block forward substitution)
#pragma unroll
                for (int i = 0; i < TPW; ++i) {
                    const int q = q0 + i * K;                     // group index within the panel
                    if (i >= ni || q == 0) continue;
                    const int row = j0 + 32 * q + 8 * warp + g;
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
            if (!waitedA) cluster_wait();       // a CTA without groups in this panel
            fence_proxy_async_all();            // the factor written above is read by the TMA of every CTA next panel
            cluster_arrive();                   // barrier B ("panel done")
            cluster_wait();
            fence_proxy_async_all();
        }

        // ---------------- z = L^-1 b sits in row R (+r);  v1 = z'z = w1' S1 w1   (:574)
        double zz = 0.0;
        for (int j = tid; j < Nr; j += CC_THREADS) {
            const double z = j < N ? S[(long long)R * ld + j] : 0.0;
            zs[j] = z;
            zz = fma(z, z, zz);
            if constexpr (NRHS == 2) zs[Nr + j] = j < N ? S[(long long)(R + 1) * ld + j] : 0.0;
        }
        const double v1 = block_sum(zz, scratch);

        // ---------------- back substitution L' x = z, right-looking over 32-column blocks (block b: CTA b mod K)
        const int nblk = Nr / NB;
        auto load_diag = [&](int b) {
            const int j0 = NB * b;
            for (int i = warp; i < NB; i += CC_WARPS) {
                const int row = j0 + i, col = j0 + lane;
                double v;
                if (row < N && col < N) v = lane <= i ? S[(long long)row * ld + col] : 0.0;
                else v = i == lane ? 1.0 : 0.0;
                P[i * LDQ + lane] = v;
            }
        };
        if (rank == (nblk - 1) % K) load_diag(nblk - 1);
        for (int b = nblk - 1; b >= 0; --b) {
            const int j0 = NB * b;
            if (rank == b % K) {
                __syncthreads();                              // P and the running right-hand side are complete
                if (warp < NRHS) {
                    double r = zs[warp * Nr + j0 + lane];
                    const double rd = 1.0 / P[lane * LDQ + lane];
#pragma unroll
                    for (int k = NB - 1; k >= 0; --k) {
                        const double xk = __shfl_sync(0xffffffffu, r * rd, k);
                        if (lane == k) r = xk;
                        if (lane < k) r = fma(-P[k * LDQ + lane], xk, r);
                    }
                    for (int peer = 0; peer < K; ++peer) cluster.map_shared_rank(xsol, peer)[warp * Nr + j0 + lane] = r;
                }
                if (K == 1) __syncthreads();                  // the same CTA refills P below
            }
            if (b > 0 && rank == (b - 1) % K) load_diag(b - 1);     // ahead of the barrier: independent of x_b
            cluster_arrive();
            cluster_wait();
            // my blocks bb < b: z_bb -= L[rows of b, columns of bb]' x_b, one warp per block
            for (int bb = rank + K * warp; bb < b; bb += K * CC_WARPS) {
                const int col = NB * bb + lane;
                double a0[NRHS], a1[NRHS];
#pragma unroll
                for (int r = 0; r < NRHS; ++r) a0[r] = a1[r] = 0.0;
                const int rows = min(NB, N - j0);
#pragma unroll 4
                for (int i = 0; i + 1 < rows; i += 2) {
                    const double l0 = S[(long long)(j0 + i) * ld + col], l1 = S[(long long)(j0 + i + 1) * ld + col];
#pragma unroll
                    for (int r = 0; r < NRHS; ++r) {
                        a0[r] = fma(l0, xsol[r * Nr + j0 + i], a0[r]);
                        a1[r] = fma(l1, xsol[r * Nr + j0 + i + 1], a1[r]);
                    }
                }
                if (rows & 1) {
                    const double l0 = S[(long long)(j0 + rows - 1) * ld + col];
#pragma unroll
                    for (int r = 0; r < NRHS; ++r) a0[r] = fma(l0, xsol[r * Nr + j0 + rows - 1], a0[r]);
                }
#pragma unroll
                for (int r = 0; r < NRHS; ++r) zs[r * Nr + col] -= a0[r] + a1[r];
            }
        }
        // every CTA reports its first failing pivot to rank 0
        if (tid == 0) cluster.map_shared_rank(fail_all, 0)[rank] = fail_s;
        cluster_arrive();
        cluster_wait();

        // ---------------- posterior scalars and weights (rank 0; its xsol holds the whole solution)
        if (rank == 0) {
            double* scal = p.scal + (long long)w * BP_S_COUNT;
            if constexpr (NRHS == 2) {
                // Jorion's Bayes-Stein estimator (:851-895) from y = C^-1 t and z = C^-1 1: see jorion_math.cuh
                const double* y = xsol;
                const double* z = xsol + Nr;
                double sy = 0.0, sz = 0.0, ty = 0.0;
                for (int j = tid; j < N; j += CC_THREADS) {
                    sy += y[j];
                    sz += z[j];
                    ty = fma(rhs[j], y[j], ty);
                }
                sy = block_sum(sy, scratch);
                sz = block_sum(sz, scratch);
                ty = block_sum(ty, scratch);
                const JorionCoef jc = jorion_coefficients(sy, sz, ty, (double)p.n_returns, (double)N);
                for (int j = tid; j < p.ldv; j += CC_THREADS) {
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
                for (int j = tid; j < p.ldv; j += CC_THREADS) {
                    const double wv = j < N ? xsol[j] : 0.0;
                    const double nu = p.mode == BP_MODE_CONJUGATE ? (wv * mult) : wv;
                    p.w1[(long long)w * p.ldv + j] = wv;
                    p.nu[(long long)w * p.ldv + j] = nu;
                    p.weights[(long long)w * p.ldv + j] = p.inv_gamma * nu;
                }
            }
            if (tid == 0) {
                int f = 0;
                for (int r = 0; r < K; ++r)
                    if (fail_all[r] != 0 && (f == 0 || fail_all[r] < f)) f = fail_all[r];
                scal[BP_S_V1] = v1;
                p.status[w] = f;
            }
        }
        __syncthreads();       // zs / xsol / fail_s are reused by the next window
    }
    // no CTA may exit while a peer can still address its shared memory
    cluster_arrive();
    cluster_wait();
}

namespace {

int env_int(const char* name, int dflt, int lo, int hi) {
    const char* e = getenv(name);
    if (!e) return dflt;
    const int v = atoi(e);
    return v >= lo && v <= hi ? v : dflt;
}

}  // namespace

// CTAs per cluster for a launch of n_windows.  Measured on the B200 (full C2 launch, 4,150 windows): splitting a window
// over a cluster cuts the DRAM traffic (5.4 instead of 10.7 MB of reads per window at K = 4) but the serial parts of a
// factorisation (diagonal blocks, the back-substitution chain) idle the other K-1 CTAs, and at N = 500 there are too
// few 32-row groups per panel to hide that: 11.8 ms (K = 1, chol_solve_kernel) / 13.6 (K = 2) / 17.8 (K = 4) / 27.6
// (K = 8).  Throughput-bound launches therefore stay with one CTA per window; the cluster kernel takes the launches
// that cannot fill the machine (a single façade window, the Jeffreys base windows of a date-range shard), where it
// shortens the latency of the launch roughly K-fold.  BP_CHOL_CLUSTER=k forces k (0 = never).
int chol_cluster_size(int n_windows, int cta_slots) {
    static const int forced = env_int("BP_CHOL_CLUSTER", -1, 0, CC_MAX_CLUSTER);
    if (forced >= 0) return forced;
    static const int slack_pct = env_int("BP_CHOL_CLUSTER_SLACK_PCT", 100, 100, 400);
    int k = CC_MAX_CLUSTER;
    while (k > 1 && (long long)n_windows * k * 100 > (long long)cta_slots * slack_pct) k >>= 1;
    return k > 1 ? k : 0;
}

size_t chol_cluster_smem_bytes(int n_assets, int nrhs) {
    const int Nr = (n_assets + NB - 1) / NB * NB;
    // zs and xsol alias the stage ring: it must hold them
    if ((size_t)CC_STAGES * CC_STAGE_BYTES < sizeof(double) * 2 * (size_t)Nr * nrhs) return 0;
    return (size_t)CC_TMA_SMEM + sizeof(double) * (size_t)(NB * LDQ + 40);
}

// Windows in flight (= resident clusters) of a launch with clusters of k CTAs; 0 if the kernel cannot run this shape
template <int NRHS>
static int cluster_capacity(int k, size_t smem, cudaLaunchConfig_t* cfg, cudaLaunchAttribute* attr) {
    if (cudaFuncSetAttribute(chol_cluster_kernel<NRHS>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess) {
        cudaGetLastError();
        return 0;
    }
    attr->id = cudaLaunchAttributeClusterDimension;
    attr->val.clusterDim.x = k;
    attr->val.clusterDim.y = 1;
    attr->val.clusterDim.z = 1;
    cfg->gridDim = dim3(k, 1, 1);
    cfg->blockDim = dim3(CC_THREADS, 1, 1);
    cfg->dynamicSmemBytes = smem;
    cfg->attrs = attr;
    cfg->numAttrs = 1;
    int n = 0;
    if (cudaOccupancyMaxActiveClusters(&n, chol_cluster_kernel<NRHS>, cfg) != cudaSuccess) {
        cudaGetLastError();
        return 0;
    }
    return n;
}

// Returns cudaErrorNotSupported when the shape does not fit (the caller falls back to chol_solve_kernel)
cudaError_t launch_chol_cluster(const SolveParams& p, const CUtensorMap& smap, int cta_slots, cudaStream_t st) {
    if (p.n_windows <= 0) return cudaSuccess;
    const int k = chol_cluster_size(p.n_windows, cta_slots);
    const int nrhs = p.estimator == BP_EST_JORION ? 2 : 1;
    const size_t smem = chol_cluster_smem_bytes(p.n_assets, nrhs);
    if (k <= 0 || smem == 0) return cudaErrorNotSupported;
    static int cap[3] = {-1, -1, -1};
    cudaLaunchConfig_t cfg{};
    cudaLaunchAttribute attr{};
    cfg.stream = st;
    const int c = nrhs == 2 ? cluster_capacity<2>(k, smem, &cfg, &attr) : cluster_capacity<1>(k, smem, &cfg, &attr);
    if (cap[nrhs] != c) {
        cap[nrhs] = c;
        if (getenv("BP_CHOL_VERBOSE")) fprintf(stderr, "[chol cluster] k=%d nrhs=%d resident clusters=%d smem=%zu\n", k, nrhs, c, smem);
    }
    if (c <= 0) return cudaErrorNotSupported;
    const int limit = env_int("BP_CHOL_MAX_CLUSTERS", c, 1, c);
    const int nclusters = p.n_windows < limit ? p.n_windows : limit;
    cfg.gridDim = dim3((unsigned)(nclusters * k), 1, 1);
    cfg.stream = st;
    cudaError_t e = nrhs == 2 ? cudaLaunchKernelEx(&cfg, chol_cluster_kernel<2>, smap, p)
                              : cudaLaunchKernelEx(&cfg, chol_cluster_kernel<1>, smap, p);
    return e != cudaSuccess ? e : cudaGetLastError();
}

}  // namespace bp
