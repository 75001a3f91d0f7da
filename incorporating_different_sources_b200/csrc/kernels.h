// Internal launch interfaces shared by the .cu translation units (not part of the C-ABI).
#pragma once
#include <cuda.h>
#include <cuda_runtime.h>
#include <cstddef>
#include <cstdint>

namespace bp {

enum { BP_MODE_CONJUGATE = 0, BP_MODE_JEFFREYS = 1 };
enum { BP_PRIOR_VW = 0, BP_PRIOR_EW = 1 };
// sibling estimators on the sample moments of the daily window (SURVEY 8(f) rank 3); they run as
// BP_MODE_JEFFREYS batches whose Gram epilogue centres with 1/m (m = n-1 returns) instead of 1/n
enum { BP_EST_NONE = 0, BP_EST_JORION = 1, BP_EST_SHRINKAGE = 2 };

// per-window scalar record written by window_prep_kernel / chol_solve_kernel
enum {
    BP_S_N0 = 0,     // conjugate prior n            (:265)
    BP_S_N1 = 1,     // posterior n                  (:282)
    BP_S_ALPHA = 2,  // n0 * m/(m-1): scale of the raw HF Gram inside S0
    BP_S_BETA = 3,   // rank-1 coefficient of the Gram epilogue (alpha*m, or 1/n for Jeffreys)
    BP_S_C = 4,      // conjugate c                  (:415-418)
    BP_S_V0 = 5,     // w0' S0 w0                    (:78)
    BP_S_M = 6,      // HF returns in the window
    BP_S_SUMA = 7,   // sum_k a_k
    BP_S_V1 = 8,     // w1' S1 w1                    (:574)
    BP_S_MCM_AVG = 9,  // average MCM over the window (:112)
    BP_S_ANORM1 = 10,  // 1-norm of the factorised matrix (condition estimate on, chol_rcond.cu)
    BP_S_RCOND = 11,   // dpocon's reciprocal 1-norm condition estimate (condition estimate on, chol_rcond.cu)
    BP_S_COUNT = 12,
    // estimator batches reuse the slots the Jeffreys path leaves at zero (slot 3 stays the Gram's beta)
    BP_S_JORION_MU_G = 0,          // grand mean mu_g                     (:882)
    BP_S_JORION_LAMBDA = 1,        // lambda_hat                          (:885)
    BP_S_JORION_V = 2,             // v_hat                               (:887)
    BP_S_JORION_Q = 4,             // (mu_hat - mu_g 1)' V_bar^-1 (mu_hat - mu_g 1)
    BP_S_JORION_ONE_VINV_ONE = 5,  // 1' V_bar^-1 1
    BP_S_LW_SHRINKAGE = 0,         // Ledoit-Wolf shrinkage intensity
    BP_S_LW_MU = 1,                // trace(emp_cov) / N
    BP_S_LW_BETA = 2,              // sklearn's beta (before the min with delta)
    BP_S_LW_DELTA = 4              // sklearn's delta
};

struct PrepParams {
    int mode;            // BP_MODE_*
    int n_assets;        // N
    int n_window;        // rolling_window n (prices); n-1 returns
    int ld;              // leading dimension of the market matrices
    int ldv;             // leading dimension of the per-window vectors
    int prior_kind;      // BP_PRIOR_*
    double mcm_scaling;
    const double* lr_daily;   // [D][ld] daily log returns (row r = log(P_r / P_{r-1}))
    const double* lr_hf;      // [R][ld] intraday log returns (dropped rows are zero rows)
    const unsigned char* hf_keep;   // [R] 1 = the return row is kept (dropna, :314), 0 = dropped
    const double* caps;       // [D][ld_caps] (dense upload layout)
    int ld_caps;
    const double* mcm;        // [D]
    int mcm_rows;             // observations averaged (min(n, available), :112)
    const double* prior_n;    // [W] injected conjugate_prior_n (nullptr: from the MCM series)
    const double* rf_row;     // [D] risk-free forward-filled onto the daily rows
    const int* day_row;       // [W] last shared return row of the window (the trade date's row for daily windows)
    const int* extra_row;     // [W] per-date last return row of resampled (weekly) windows, or nullptr
    const int* caps_row;      // [W] row of the trade date in the caps matrix, or nullptr (= day_row)
    const int* span_days;     // [W]
    const int* hf_row0;       // [W] first intraday RETURN row of the HF window (= first price row + 1)
    const int* hf_span;       // [W] HF return rows the window spans; m = the kept rows among them
    double* t;                // [W][ldv]
    double* pvec;             // [W][ldv]  u - a'a/2
    double* gvec;             // [W][ldv]  hbar (conjugate) or t (Jeffreys)
    double* rhs;              // [W][ldv]  b = c S0 w0 + t   (or t)
    double* w0;               // [W][ldv]
    double* s0w0;             // [W][ldv]
    double* scal;             // [W][BP_NSCAL]
    double* y_ws;             // [W][y_stride] scratch for the HF row dots
    long long y_stride;
    // banded-GEMM form of the daily pass (band_prep.cu), used for batches of consecutive trade dates
    // Pre-summed intraday day blocks (long HF look-backs, bp_api.cu "presum"): the window's column sums come from the
    // scanned per-day column sums instead of a pass over its own rows, and S0 w0 / v0 / c / rhs are finished by
    // conj_post_kernel from the mat-vec partials the Gram kernel leaves behind
    int hf_presum;
    const double* hf_vsum;    // [3 nb][ld]: suffix' sums at nb + b, prefix sums at 2 nb + b (same ids as the tile store)
    const int* hf_vids;       // [W][3] ids into hf_vsum (-1 = absent)
    int beta_den;             // Jeffreys-mode rank-1 coefficient beta = 1 / beta_den (0: n_window, :600; estimators: n-1)
    int use_band;
    double* band_aw;          // [W][band_ld] risk-free weights a_k(w)
    int band_ld;
    double* band_stats;       // [W][2] sum a, sum a^2
};

// Per-window job descriptor of the Gram kernel (GRAM_DESC_INTS ints), 10 per phase (A = intraday, scaled by
// alpha, at offset 0; B = daily at offset 10):
//   [0] K0.row0 [1] K0.rows  [2] K1.row0 [3] K1.rows      head / tail rows contracted on the tensor cores
//   [4] coarse.block0 [5] coarse.nblocks                   whole coarse blocks, added from the coarse tile store
//   [6] fineA.block0  [7] fineA.nblocks                    whole fine blocks between the head rows and the coarse blocks
//   [8] fineB.block0  [9] fineB.nblocks                    whole fine blocks between the coarse blocks and the tail rows
constexpr int GRAM_DESC_INTS = 20;
constexpr int GRAM_PHASE_INTS = 10;
constexpr int GRAM_BLOCK_TILE_DOUBLES = 128 * 128;   // one stored 128x128 tile, fragment-major

struct GramParams {
    int n_windows;
    int w_stride;        // job window q works on window q * w_stride of every per-window array (0 = 1); the Jeffreys
                         // chain path computes the Gram of the base windows only
    int n_assets;        // N
    int ldS;             // leading dimension of the output matrices
    long long win_stride;    // doubles between consecutive output matrices
    int ldv;
    int mirror;          // also write the upper triangle
    const int* desc;         // [W][GRAM_DESC_INTS]
    int use_phaseA;          // contract / add the intraday phase (tensor map 0, storeA)
    int use_phaseB;          // contract / add the daily phase (tensor map 1, storeB)
    // block tile stores [phase][level 0 = coarse, 1 = fine]: tile (block b, pair p) at
    // ((b * npairs) + p) * GRAM_BLOCK_TILE_DOUBLES
    const double* store[2][2];
    int tile_store_out;      // 1: block precompute, write raw accumulators fragment-major to out[(w*npairs+pair)*tile]
    const double* scal;      // [W][BP_S_COUNT] (alpha, beta)
    int use_alpha;
    int use_beta;
    const double* pvec;      // [W][ldv] or nullptr
    const double* gvec;      // [W][ldv] or nullptr
    double* out;             // [W][win_stride]  (or the tile store in tile_store_out mode)
    // optional by-product of phase A: the raw intraday Gram times the prior weights, G w0, as per-tile partial sums
    // mv_part[((w * npairs + pair) * 2 + dir) * 128 + k]: dir 0 = rows of tile row ti (sum over the tile's columns),
    // dir 1 = columns of tile column tj (sum over the tile's rows; off-diagonal tiles only).  Reduced in a fixed
    // order by conj_post_kernel: no atomics, bit-reproducible.
    double* mv_part;
    const double* mv_w0;     // [W][ldv] prior weights
};

// S0 w0 = alpha (G w0 - m hbar (hbar'w0)), v0 = w0'S0w0 (:64-88), c (:415-418), rhs = c S0w0 + t (:489) from the
// mat-vec partials of the Gram kernel (pre-summed day blocks: no pass over the window's own intraday rows)
struct PostParams {
    int n_windows, n_assets, ldv;
    const double* mv_part;   // [W][npairs][2][128]
    const double* w0;        // [W][ldv]
    const double* gvec;      // [W][ldv] hbar
    const double* t;         // [W][ldv]
    double* s0w0;            // [W][ldv]
    double* rhs;             // [W][ldv]
    double* scal;            // [W][BP_S_COUNT] reads n0, alpha, m; writes c, v0
};
cudaError_t launch_conj_post(const PostParams& p, cudaStream_t st);
// column sums of the inner rows (all but the first) of every block: out[b][ld], blocks given by starts[b], starts[b+1]
void launch_block_col_sums(const double* M, int ld, const int* starts, int b0, int b1, double* out, cudaStream_t st);
// Scans over chunks of `chunk` consecutive blocks (suffix' at nb + b, prefix at 2 nb + b, see bp_api.cu):
//   FD[b] = inner[b] + overnight[b] (vectors) or inner tile + overnight (x) overnight (tiles)
//   prefix[b]  = FD[chunk start] + ... + FD[b]          suffix'[b] = inner[b] + FD[b+1] + ... + FD[chunk end]
void launch_vec_scan(double* vsum, int ld, const double* M, const int* starts, int nb, int chunk, cudaStream_t st);
void launch_tile_scan(double* store, int npairs, int n_tiles_side, const double* M, int ld, const int* starts, int nb,
                      int chunk, cudaStream_t st);
// per-window blocks of rows and columns stacked into one dense [sum rows][n] matrix; rows = [W][3] (first pool row,
// first stack row, row count), cols = [W][n] or nullptr (columns 0..n-1); max_rows = the largest row count.  Any n.
void launch_gather_window_blocks(const double* src, long long ld_src, double* dst, int n, int n_windows, const int* cols,
                                 const long long* rows, long long max_rows, cudaStream_t st);
void launch_gather_rows_indexed(double* M, int ld, const int* src_rows, long long dst_row0, int k0, int k1, cudaStream_t st);

struct SolveParams {
    int n_windows;
    int w_stride;            // CTA job q factorises window q * w_stride (0 = 1), see GramParams::w_stride
    int n_assets;
    int ldS;
    long long win_stride;
    int ldv;
    int mode;                // BP_MODE_*
    int estimator;           // BP_EST_*: JORION solves two right-hand sides (t and 1) and combines them (:851-895)
    int n_returns;           // m = n - 1 (Jorion's T)
    double inv_gamma;        // 1 / risk_aversion
    double* S;               // [W][win_stride] in: lower triangle of S1 / J ; out: Cholesky factor
    const double* rhs;       // [W][ldv]
    double* scal;            // [W][BP_NSCAL]  (reads n1, writes v1)
    double* w1;              // [W][ldv] posterior w  (S^-1 rhs)
    double* nu;              // [W][ldv]
    double* weights;         // [W][ldv]
    int* status;             // [W] 0 = ok, k+1 = non-positive pivot at column k
    long long* debug;        // optional phase-cycle counters (BP_CHOL_PROFILE), normally nullptr
};

// Row R of the solver workspace at which the right-hand side(s) ride along through the factorisation (rows R .. R+nrhs-1,
// so that L z = b comes out as row R of the factor).  R = roundup(N, 8): for N mod 32 in 1..24 that is a padding row at
// most Nr - 8 (Nr = roundup(N, 32)), so up to 8 right-hand sides fit below Nr and the panels end at row Nr - 1;
// otherwise R = Nr and the panels cover the extra m-tile Nr .. Nr+7 (the workspace has ldS + 8 rows for it).
__host__ __device__ constexpr int chol_rhs_row(int n_assets) { return (n_assets + 7) / 8 * 8; }

struct DenseParams {
    int n_assets, ldS, ldv, n_window;
    double n0, n1, c_in;
    int has_c;
    const double* T;       // [N][N] dense
    const double* t;       // [N]
    const double* S0;      // [N][N] dense
    const double* w0;      // [N]
    const double* S1_in;   // [N][N] dense or nullptr
    double* s0w0;          // [N]
    double* rhs;           // [ldv]
    double* S_out;         // padded [rows][ldS]
    double* scal;          // [BP_S_COUNT]
};

struct LoopParams {
    int n_assets, n_rebalances;
    int ldw;                     // leading dimension of weights
    const double* weights;       // [R][ldw] weights chosen at each rebalance (0 for non-members)
    const unsigned char* member; // [R][N] membership of the rebalance universe, or nullptr (= all)
    const int* reb_row;          // [R] daily row of each rebalance date (ascending)
    int last_row;                // daily row of the last backtest date (>= reb_row[R-1])
    const double* prices;        // dense [D][ld_prices]
    int ld_prices;
    const double* caps;          // dense [D][ld_caps]
    int ld_caps;
    const double* rf_row;        // [D]
    double distance_scale;       // risk_aversion (or 1) — the reference scales the weights before comparing (:1101-1102)
    double turnover_cost_bps;
    double* returns;             // [last_row - reb_row[0]] one per trading day after the first rebalance
    double* turnover;            // [R-1]
    double* metrics;             // [R][5]
};
cudaError_t launch_backtest_loop(const LoopParams& p, cudaStream_t st);

// evaluation statistics of a path ensemble (eval_kernels.cu); the BP_PM_* indices are declared in bayes_portfolio.h
struct PathMetricsParams {
    int n_paths, n_obs;
    long long ld;                // row stride of returns / excess
    const double* returns;       // [P][ld] simple returns
    const double* excess;        // [P][ld] excess simple returns (compute_excess_returns, :703-719)
    double years;                // (index[-1] - index[0]).days / 365  (CAGR, :520-524)
    double* out;                 // [P][BP_PM_COUNT]
};
cudaError_t launch_path_metrics(const PathMetricsParams& p, cudaStream_t st);

void launch_gather_log_returns(const double* P, int ld_in, const int* num, const int* den, double* out, int ld_out,
                               int rows, int n_assets, cudaStream_t st);
void launch_range_sum(const double* store, const int* ranges, int n_ranges, int npairs, double* out, cudaStream_t st);
void launch_combine_runs(const double* rs_coarse, const double* rs_fine, const int* triples, int n, int npairs,
                         double* out, cudaStream_t st);
void launch_fetch_ints(const int* src_host, int* dst, long long n, cudaStream_t st);
void launch_excess_returns(const double* lr, int ld, const double* rf_row, int day_row, int span_days, int n_window,
                           int N, double* X, cudaStream_t st);
void launch_dense_prep(const DenseParams& p, bool jeffreys, cudaStream_t st);
void launch_quadform(const double* S, int ldS, const double* w, int N, double* v_out, double n1, double inv_gamma,
                     double* nu, double* weights, cudaStream_t st);
void launch_log_returns(const double* P, int ld_in, double* out, int ld_out, long long rows, int n_assets,
                        int sm_count, cudaStream_t st, long long row_begin = 0);
// intraday rows [row_begin, rows): returns with the reference's dropna, keep[r] = 1 for a kept row (stream_kernels.cu)
void launch_hf_log_returns(const double* P, int ld_in, double* out, int ld_out, unsigned char* keep, long long row_begin,
                           long long rows, int n_assets, int sm_count, cudaStream_t st);
size_t prep_smem_bytes(int n_window, int ldv);
cudaError_t launch_window_prep(const PrepParams& p, int n_windows, cudaStream_t st, long long n_daily_rows = 0);
cudaError_t launch_daily_band(const PrepParams& p, int n_windows, long long n_rows, cudaStream_t st);
void launch_unpack_sym(const double* S, long long win_stride, int ldS, int N, int W, double* out, cudaStream_t st);
void launch_unpack_vec(const double* v, int ldv, int N, long long W, double* out, cudaStream_t st);

// Gram (DMMA + TMA)
constexpr int GRAM_KT = 32;        // rows per TMA k-tile
constexpr int GRAM_TILE = 128;     // output tile edge
cudaError_t launch_gram(const GramParams& p, const CUtensorMap& map0, const CUtensorMap& map1, int sm_count,
                        cudaStream_t st);
// Ledoit-Wolf shrinkage of the centred Gram C = X_c'X_c in the solver workspace (in place), s the shrinkage intensity:
// S <- C + rho I, rhs <- t / (1 - s), rho = s mu m / (1 - s): Sigma_LW w = mu_hat scaled by m / (1 - s) (sklearn.covariance.ledoit_wolf
// as called by pypfopt's CovarianceShrinkage.ledoit_wolf(), portfolio_calculations.py:727-729).  s = 0 for N = 1; a clipped
// window (s = 1, Sigma_LW = mu I) gets S <- mu m I (lower triangle) and rhs <- t
struct ShrinkParams {
    int n_windows, n_assets, n_window, ld, ldv, ldS;
    long long win_stride;
    const double* lr_daily;   // [D][ld]
    const double* rf_row;     // [D]
    const int* day_row;       // [W]
    const int* extra_row;     // [W] or nullptr
    const int* span_days;     // [W]
    const double* t;          // [W][ldv]
    double* S;                // [W][win_stride] lower triangle of C, diagonal overwritten
    double* rhs;              // [W][ldv] right-hand side of the solve, overwritten
    double* scal;             // [W][BP_S_COUNT]
};
cudaError_t launch_lw_shrink(const ShrinkParams& p, cudaStream_t st);
// Jeffreys windows of consecutive trade dates relative to a factorised base window (jeffreys_chain.cu)
struct ChainParams {
    int n_windows;           // W, consecutive trade dates: day_row[w] = day_row[0] + w
    int group;               // windows per group; window g * group is the base (factor in its S slot)
    int n_assets, n_window, ld, ldv, ldS;
    int estimator;           // BP_EST_NONE: Jeffreys (J = T - tt'/n, :600); BP_EST_JORION: C = T - tt'/m, m = n-1, and the
                             // Bayes-Stein combination of C^-1 t and C^-1 1 (:851-895)
    long long win_stride;
    double inv_gamma;
    const double* lr_daily;  // [D][ld]
    const int* day_row;      // [W]
    const double* S;         // [W][win_stride]: the base slots hold the Cholesky factor of J_base
    const double* t;         // [W][ldv]
    const double* pvec;      // [W][ldv]
    double* w1;              // [W][ldv]
    double* nu;
    double* weights;
    double* scal;            // [W][BP_S_COUNT] (writes v1)
    int* status;             // [W] reads the base's flag, writes the chained windows': the base's flag when it is
                             // non-zero, else N+1 for a window singular relative to the base (pivot <= 2^-40 max |M|)
                             // or with v1 <= 0 (Jorion: t'C^-1 t <= 0), else 0
};
size_t chain_smem_bytes(int n_assets);
int chain_max_group();
cudaError_t launch_jeffreys_chain(const ChainParams& p, cudaStream_t st);
cudaError_t launch_chol_solve(const SolveParams& p, const CUtensorMap& smap, int sm_count, cudaStream_t st);
int chol_wave_windows(int sm_count);
// dynamic shared memory of chol_solve_kernel for N assets and nrhs right-hand sides; 0 if N is too large for the
// back-substitution vectors, which alias the TMA stage ring
size_t chol_smem_bytes(int n_assets, int nrhs);
// largest N the solver accepts with nrhs right-hand sides (3072 for one, 1536 for Jorion's two): the callers check it
// before any upload or launch
int chol_max_assets(int nrhs);
// chol_cluster.cu: one thread-block cluster of K CTAs per window for launches of fewer than cta_slots / 2 windows (K =
// 8, 4 or 2, the largest with n_windows * K <= cta_slots); cudaErrorNotSupported otherwise (and when N is too large for
// the aliased back-substitution vectors, or with BP_CHOL_CLUSTER=0): the caller then runs chol_solve_kernel
cudaError_t launch_chol_cluster(const SolveParams& p, const CUtensorMap& smap, int cta_slots, cudaStream_t st);
// chol_rcond.cu, the condition estimate of the windows of a solve launch (same n_windows, w_stride, S, scal, status):
// launch_sym_norm1 before the factorisation writes anorm1 of the lower triangle of S to scal[BP_S_ANORM1];
// launch_chol_rcond after it reads the factor, the status and anorm1 and writes scal[BP_S_RCOND]
cudaError_t launch_sym_norm1(const SolveParams& p, cudaStream_t st);
cudaError_t launch_chol_rcond(const SolveParams& p, cudaStream_t st);

}  // namespace bp
