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
// The arithmetic of U's start and padding, F, T, the back substitution and the epilogue is the shared code of
// chol_panel.cuh, so that chol_cluster_kernel gives the same bits; this file holds the slab schedule.
//
// k-permutation: inside a 16-column chunk, DMMA step q contracts columns {2q, 2q+1, 8+2q, 9+2q}
// over the four tig lanes.  With the 128-byte swizzle (16-byte unit index XOR row&7) the 16 lanes of
// a half warp then hit 16 distinct 8-byte words of the 128-byte bank line: every LDS.64 fragment
// load is conflict free.  A and B fragments use the same assignment, so the contraction is exact.
#include <cstdio>
#include <cstdlib>

#include "chol_panel.cuh"

namespace bp {

using namespace chol;

#ifndef CH_NWARPS
#define CH_NWARPS 4
#endif
constexpr int CH_WARPS = CH_NWARPS;                 // warps per window (CTA)
#ifndef CH_CTAS_PER_SM
#define CH_CTAS_PER_SM 6
#endif
constexpr int CH_OCC = CH_CTAS_PER_SM;              // resident CTAs (windows) per SM
constexpr int CH_THREADS = CH_WARPS * 32;

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
constexpr int CH_STAGE_BYTES = (ABOXES + 1) * BOX_BYTES;   // A slab + 1 B box
constexpr int CH_TMA_SMEM = CH_STAGES * CH_STAGE_BYTES + 1024;

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

    if (tid == 0) init_tma_ring<CH_STAGES, CH_WARPS>(&smap, full_bar, empty_bar);
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
        // the right-hand side(s) ride along as rows R (, R+1) of S
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

                double acc[TPW][4][2];     // m-tile i of this warp: row j0 + 8 (slab0 + warp + CH_WARPS i) + g
#pragma unroll
                for (int i = 0; i < TPW; ++i)
                    tile_start<NRHS, true>(acc[i], j0 + 8 * (slab0 + warp + CH_WARPS * i) + g, i < ni, S, ld, rhs, N, R, j0, tig);

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

                if (slab_row + 8 * slab_tiles > N || j0 + NB > N) {
#pragma unroll
                    for (int i = 0; i < TPW; ++i)
                        tile_fix_padding<NRHS>(acc[i], j0 + 8 * (slab0 + warp + CH_WARPS * i) + g, N, R, j0, tig);
                }

                if (slab0 == 0) {
                    // ---------------- F: warp q < 4 holds row block q of the diagonal block in acc[0]
                    PROF(0)
                    factor_diag_block(acc[0], P, fail_s, j0, N, warp, lane);
                    PROF(1)
                    store_diag_block<NRHS, CH_WARPS>(S, ld, P, j0, N, R, warp, lane);
                }
                // ---------------- T: the m-tiles below the diagonal block
#pragma unroll
                for (int i = 0; i < TPW; ++i) {
                    const int q = slab0 + warp + CH_WARPS * i;     // m-tile index within the panel
                    if (i >= ni || q < NB / 8) continue;
                    tile_solve<NRHS>(acc[i], P, S, ld, j0 + 8 * q + g, N, R, j0, g, tig);
                }
            }
            fence_proxy_async_all();        // the factor written above is read by TMA in the next panels
            __syncthreads();
            PROF(2)
        }

        const double v1 = load_z<NRHS, CH_THREADS>(xs, S, ld, N, Nr, R, scratch);

        // ---------------- back substitution, in place in xs
        for (int b = Nr / NB - 1; b >= 0; --b) {
            load_diag_block<CH_WARPS>(P, S, ld, b, N, warp, lane);
            __syncthreads();
            if (warp < NRHS) {
                double* x = xs + warp * Nr + NB * b + lane;
                *x = solve_diag_block(*x, P, lane);
            }
            __syncthreads();
            for (int bb = warp; bb < b; bb += CH_WARPS) reduce_block<NRHS>(xs, xs, S, ld, Nr, N, b, NB * bb + lane);
        }
        __syncthreads();

        PROF(3)
        write_outputs<NRHS, CH_THREADS>(p, w, xs, Nr, v1, fail_s, scratch);
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
