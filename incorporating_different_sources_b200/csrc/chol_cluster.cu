// Batched blocked Cholesky + triangular solves + posterior scalars, ONE THREAD-BLOCK CLUSTER PER WINDOW.
//
// The factorisation of chol_solve_kernel (left-looking, 32-column panels, TMA-fed DMMA panel update with the panel
// solve fused into its epilogue, register-level 32x32 diagonal block, right-hand side(s) riding along as rows R, R+1;
// w1 = inv(S1)(c S0 w0 + t) :485-489, nu :572-575, Jeffreys :600-606, weights = (1/gamma) nu :836,:849), but the rows
// of a window are spread over the K CTAs of a cluster instead of one CTA doing everything.  All arithmetic is the
// shared code of chol_panel.cuh, so that both kernels give the same bits; this file holds the cluster's schedule.
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

#include "chol_panel.cuh"

namespace cg = cooperative_groups;

namespace bp {

using namespace chol;

namespace {

constexpr int CC_WARPS = 4;
constexpr int CC_THREADS = CC_WARPS * 32;
#ifndef CC_CTAS_PER_SM
#define CC_CTAS_PER_SM 6
#endif
constexpr int CC_OCC = CC_CTAS_PER_SM;
constexpr int TPW = 2;                               // groups (A boxes) per pass = m-tiles per warp and pass
constexpr int CC_STAGES = 2;
constexpr int CC_STAGE_BYTES = (TPW + 1) * BOX_BYTES;   // A boxes + 1 B box
constexpr int CC_TMA_SMEM = CC_STAGES * CC_STAGE_BYTES + 1024;
constexpr int CC_MAX_CLUSTER = 8;

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
    const int R = chol_rhs_row(N);             // row index of the right-hand side
    const int rows_end = max(Nr, R + 8);       // the panels cover rows j0 .. rows_end-1
    const int rowsS = (int)(p.win_stride / ld);
    const int stride = max(p.w_stride, 1);
    // back substitution vectors alias the TMA stages (idle after the last panel): running rhs and solution
    double* zs = reinterpret_cast<double*>(stage_mem);   // [NRHS][Nr]
    double* xsol = zs + NRHS * Nr;                        // [NRHS][Nr]

    if (tid == 0) init_tma_ring<CC_STAGES, CC_WARPS>(&smap, full_bar, empty_bar);
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

                double acc[TPW][4][2];     // m-tile i of this warp: row j0 + 32 (q0 + i K) + 8 warp + g
#pragma unroll
                for (int i = 0; i < TPW; ++i)
                    tile_start<NRHS, false>(acc[i], j0 + 32 * (q0 + i * K) + 8 * warp + g, i < ni, S, ld, rhs, N, R, j0, tig);

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

                if (j0 + 32 * (q0 + (nboxes - 1) * K) + 32 > N || j0 + NB > N) {
#pragma unroll
                    for (int i = 0; i < TPW; ++i)
                        tile_fix_padding<NRHS>(acc[i], j0 + 32 * (q0 + i * K) + 8 * warp + g, N, R, j0, tig);
                }

                if (q0 == 0) {
                    // ---------------- F (this CTA owns the diagonal group), packed block pushed to the peers, barrier A
                    factor_diag_block(acc[0], P, fail_s, j0, N, warp, lane);
                    for (int peer = 0; peer < K; ++peer) {
                        if (peer == rank) continue;
                        double* dst = cluster.map_shared_rank(P, peer);
                        for (int e = tid; e < NB * LDQ; e += CC_THREADS) dst[e] = P[e];
                    }
                    cluster_arrive();
                    store_diag_block<NRHS, CC_WARPS>(S, ld, P, j0, N, R, warp, lane);
                }
                if (!waitedA) {
                    cluster_wait();
                    waitedA = true;
                }
                // ---------------- T: the groups below the diagonal one
#pragma unroll
                for (int i = 0; i < TPW; ++i) {
                    const int q = q0 + i * K;                     // group index within the panel
                    if (i >= ni || q == 0) continue;
                    tile_solve<NRHS>(acc[i], P, S, ld, j0 + 32 * q + 8 * warp + g, N, R, j0, g, tig);
                }
            }
            if (!waitedA) cluster_wait();       // a CTA without groups in this panel
            fence_proxy_async_all();            // the factor written above is read by the TMA of every CTA next panel
            cluster_arrive();                   // barrier B ("panel done")
            cluster_wait();
            fence_proxy_async_all();
        }

        const double v1 = load_z<NRHS, CC_THREADS>(zs, S, ld, N, Nr, R, scratch);

        // ---------------- back substitution, right-looking over 32-column blocks (block b: CTA b mod K)
        const int nblk = Nr / NB;
        if (rank == (nblk - 1) % K) load_diag_block<CC_WARPS>(P, S, ld, nblk - 1, N, warp, lane);
        for (int b = nblk - 1; b >= 0; --b) {
            const int j0 = NB * b;
            if (rank == b % K) {
                __syncthreads();                              // P and the running right-hand side are complete
                if (warp < NRHS) {
                    const double r = solve_diag_block(zs[warp * Nr + j0 + lane], P, lane);
                    for (int peer = 0; peer < K; ++peer) cluster.map_shared_rank(xsol, peer)[warp * Nr + j0 + lane] = r;
                }
                if (K == 1) __syncthreads();                  // the same CTA refills P below
            }
            if (b > 0 && rank == (b - 1) % K) load_diag_block<CC_WARPS>(P, S, ld, b - 1, N, warp, lane);   // ahead of the barrier: independent of x_b
            cluster_arrive();
            cluster_wait();
            // my blocks bb < b, one warp per block
            for (int bb = rank + K * warp; bb < b; bb += K * CC_WARPS) reduce_block<NRHS>(zs, xsol, S, ld, Nr, N, b, NB * bb + lane);
        }
        // every CTA reports its first failing pivot to rank 0
        if (tid == 0) cluster.map_shared_rank(fail_all, 0)[rank] = fail_s;
        cluster_arrive();
        cluster_wait();

        // ---------------- posterior scalars and weights (rank 0; its xsol holds the whole solution)
        if (rank == 0) {
            int f = 0;       // the window's status: the first failing pivot over the ranks (written by thread 0)
            if (tid == 0)
                for (int r = 0; r < K; ++r)
                    if (fail_all[r] != 0 && (f == 0 || fail_all[r] < f)) f = fail_all[r];
            write_outputs<NRHS, CC_THREADS>(p, w, xsol, Nr, v1, f, scratch);
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
