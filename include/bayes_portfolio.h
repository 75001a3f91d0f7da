/* bayes_portfolio.h — C ABI of libbayes_portfolio.so (sm_100a).
 *
 * Drop-in boundary for ONE hot path of vilnik/incorporating-different-sources: the rolling-window
 * Bayesian tangency-portfolio weight computation of src/portfolio_calculations.py as driven by the
 * backtest loop (SURVEY.md §8).  The reference has no FFI of its own (pure Python); these entry
 * points are what a ctypes binding of that path binds — see INTEGRATION.md for the stub — and each
 * cites the reference interface it replaces (file:line into /root/reference/src/).
 *
 * Conventions
 *  - plain pointers and sizes only; no torch / pandas types cross this boundary;
 *  - every function returns 0 on success, non-zero on error; bp_last_error() has the message
 *    (the Python shim maps the codes onto the reference's exception types, SURVEY §8(b));
 *  - the market (prices, caps, MCM series, risk-free rate) is uploaded once and stays resident in
 *    HBM; window batches are described by integer row indices computed on the host;
 *  - OUTPUT pointers may be host pointers (pageable or pinned) or device pointers; the library
 *    detects which.  With host outputs the call returns after the data has landed; with device
 *    outputs it is asynchronous on the handle's stream;
 *  - all floating point is IEEE double; all indices are int32 row numbers into the uploaded arrays.
 */
#ifndef BAYES_PORTFOLIO_H
#define BAYES_PORTFOLIO_H

#include <stddef.h>

#ifdef __cplusplus
extern "C" {
#endif

#define BP_OK 0
#define BP_ERR_INVALID 1      /* bad argument (maps to ValueError)                                  */
#define BP_ERR_CUDA 2         /* CUDA runtime / driver failure (RuntimeError)                        */
#define BP_ERR_NO_DEVICE 3    /* no usable sm_100 device: the library never falls back to the CPU    */
#define BP_ERR_STATE 4        /* call order violated, e.g. no market uploaded                        */

#define BP_NSCAL 12           /* doubles per window in bp_outputs.scalars                            */
/* indices into the per-window scalar record */
#define BP_SCAL_N0 0          /* conjugate prior n0            portfolio_calculations.py:247-267     */
#define BP_SCAL_N1 1          /* posterior n1 = n0 + n         :269-282                              */
#define BP_SCAL_ALPHA 2       /* n0 * m/(m-1); NaN when m < 2  :317-318,:333                         */
#define BP_SCAL_BETA 3        /* rank-1 coefficient used by the Gram epilogue                       */
#define BP_SCAL_C 4           /* conjugate c                   :382-430                              */
#define BP_SCAL_V0 5          /* w0' S0 w0                     :64-88                                */
#define BP_SCAL_M 6           /* HF returns m kept by dropna   :314 (of the hf_hi - hf_lo - 1 spanned) */
#define BP_SCAL_SUMA 7        /* sum of risk-free adjustments  :48                                   */
#define BP_SCAL_V1 8          /* w1' S1 w1                     :574                                  */
#define BP_SCAL_MCM_AVG 9     /* average MCM over the window   :112                                  */
/* Condition estimate (bp_set_condition_estimate; the solver writes neither slot while it is off), for every window the solver
 * factorises.  A is the symmetric matrix of the lower triangle the solver factorises: S1 (conjugate), J (Jeffreys),
 * C (Jorion), C + rho I (shrinkage, after the Ledoit-Wolf rewrite), the caller's S (bp_solve_batched), S1
 * (bp_dense_posterior).  Windows solved relative to a base window (bp_set_jeffreys_chain) are not factorised: while
 * the estimate is on, every window is.                                                                           */
#define BP_SCAL_ANORM1 10     /* max_j sum_i |A_ij|, read before the factorisation overwrites A                   */
#define BP_SCAL_RCOND 11      /* (1 / est) / anorm1, est = dlacn2's estimate of ||A^-1||_1 (Hager-Higham, ITMAX 5,
                                 x >= 0 -> +1, first-index idamax) with A^-1 v through the window's own factor L L':
                                 what LAPACK's dpocon returns.  0 when the status is non-zero (incomplete factor),
                                 when anorm1 is 0 (or not a positive number), and when a solve has a non-finite
                                 1-norm (dpocon's overflow exit); N = 1 gives 1 / (|A^-1| anorm1).  est is a lower
                                 bound of ||A^-1||_1 up to the rounding of the solves, so rcond >= 1/cond_1.        */

/* stages reported by bp_get_stage_times */
#define BP_NSTAGE 8
#define BP_STAGE_LOGRET 0     /* prices -> log returns                  :37, :314                    */
#define BP_STAGE_PREP 1       /* per-window O(N K) reductions + scalars :40-57,:90-114,:247-282,:361-430 */
#define BP_STAGE_GRAM 2       /* batched Gram / covariance (DMMA)       :180-182, :317-318, :358, :600 */
#define BP_STAGE_SOLVE 3      /* Cholesky + solves + weights            :485-489, :572-575, :602-606  */
#define BP_STAGE_CHAIN 4      /* Jeffreys windows solved relative to a factorised base window :600-606 */
#define BP_STAGE_COND 5       /* condition estimate: anorm1 before, rcond after each factorisation      */

typedef struct bp_handle bp_handle;

/* The data the weight functions read (the frames of data_handling.py:282-291, already aligned to
 * one business-day calendar by the host).  Row-major, densely packed (leading dimension n_assets). */
typedef struct {
    int n_assets;               /* N: columns of every matrix, in the caller's column order          */
    int n_days;                 /* D: rows of prices / caps / mcm / rf_row                           */
    long long n_hf_rows;        /* R: rows of hf_prices (may be 0 for Jeffreys-only use)             */
    const double* prices;       /* [D][N] daily close           -> k_stock_prices_df                 */
    const double* caps;         /* [D][N] market caps           -> k_stock_market_caps_df (may be NULL) */
    const double* hf_prices;    /* [R][N] intraday prices       -> k_stock_intraday_prices_df        */
                                /* May hold NaN (missing bars).  As the reference's dropna (:314), intraday
                                   return row r (log of price row r over row r-1) is dropped when any of its
                                   N returns is NaN: a NaN bar in row r-1 or r of ANY column drops it.  The
                                   decision does not depend on the window; a window uses the kept rows among
                                   its own, m of them (BP_SCAL_M), and a window with m < 2 gets NaN S0, S1
                                   and weights and a non-zero status, as the reference's all-NaN cov does. */
    const double* mcm;          /* [n_mcm][D] VIX / EPU ...     -> mcm_prices_df (may be NULL)       */
    int n_mcm;
    const double* rf_row;       /* [D] annualised risk-free rate forward-filled onto the daily rows
                                   (risk_free_rate_df.reindex(method='ffill'), :54)                  */
} bp_market_desc;

/* One batch of rebalance windows sharing a portfolio_spec (portfolio_specs.py:80-90). */
typedef struct {
    int n_windows;              /* W                                                                 */
    int rolling_window;         /* spec["rolling_window"]: n prices -> n-1 returns (:159, F2)        */
    const int* day_row;         /* [W] row of trading_date_ts in the daily arrays (:145)             */
    const int* span_days;       /* [W] calendar days between first and last window date (:40-41)     */
    const int* hf_lo;           /* [W] first intraday PRICE row with ts > d - D + 1 day (:310-312)   */
    const int* hf_hi;           /* [W] one past the last intraday row with ts <= d + 1 day           */
    int mcm_index;              /* which uploaded MCM series (VIX / EPU)                             */
    double mcm_scaling;         /* spec["mcm_scaling"] (:265)                                        */
    double risk_aversion;       /* spec["risk_aversion"] (:836,:849)                                 */
    int prior_weights;          /* 0: value weighted ("vw" in strategy, :369) 1: equally weighted    */
    int mcm_rows;               /* MCM observations averaged; 0 = rolling_window (iloc[-n:], :112)   */
    const double* prior_n;      /* [W] injected conjugate_prior_n (the reference's conjugate_prior_n=
                                   argument, :289,:388,:507) or NULL: derive n0 from the MCM series  */
    int resampled;              /* 1: weekly windows (rolling_window_frequency == "weekly", :151-153): day_row
                                   and extra_row index the rows defined by bp_set_resampled              */
    const int* extra_row;       /* [W] resampled windows only: row of the window's LAST return (price at the
                                   trade date against the previous week's close); the n-2 returns before it
                                   are the shared weekly rows ending at day_row                         */
    const int* caps_row;        /* [W] resampled windows only: daily row of the trade date (market caps)  */
} bp_window_batch;

/* Resampled return rows for weekly windows (adjust_stock_prices_window / calculate_average_mcm_window with
 * resample('W').last(), :106, :153): row i is ln(P[num_row[i]] / P[den_row[i]]) of the uploaded daily prices
 * (computed on the device); rf_row / mcm give the risk-free rate (forward-filled at the row's label date,
 * :54) and the MCM observation of each row.  The host chooses the rows: one per week plus one per trade date. */
typedef struct {
    int n_rows;
    const int* num_row;         /* [n_rows] daily price row in the numerator                             */
    const int* den_row;         /* [n_rows] daily price row in the denominator (== num_row: zero row)     */
    const double* rf_row;       /* [n_rows]                                                               */
    const double* mcm;          /* [n_mcm][n_rows] (n_mcm as uploaded with the market) or NULL            */
} bp_resampled_desc;
int bp_set_resampled(bp_handle* h, const bp_resampled_desc* r);

/* Optional outputs (NULL = not wanted).  Vectors are [W][N], matrices [W][N][N] dense symmetric. */
typedef struct {
    double* weights;            /* (1/gamma) nu                  :836 / :849                         */
    double* nu;                 /* posterior mean nu             :572-575 / :606                     */
    double* w1;                 /* conjugate posterior w         :489 (Jeffreys: same as nu)         */
    double* t;                  /* canonical statistic t         :222                                */
    double* w0;                 /* prior weights                 :361-380                            */
    double* rhs;                /* c S0 w0 + t                   :489                                */
    double* scalars;            /* [W][BP_NSCAL]                                                     */
    int* status;                /* [W] 0 ok; k+1: pivot k not positive (reference would return garbage, F6).
                                   A window solved relative to a base window (bp_set_jeffreys_chain) reports its
                                   base's status when that is non-zero, else N+1 when its own matrix is singular
                                   relative to the base (a Gauss-Jordan pivot at or below 2^-40 of the largest entry
                                   of its small system) or v1 <= 0 (Jorion: t'C^-1 t <= 0), else 0. */
    double* T;                  /* canonical statistic T         :180-182                            */
    double* S0;                 /* conjugate prior S             :333                                */
    double* S1;                 /* posterior S (or Jeffreys J)   :358 / :600-601                     */
} bp_outputs;

const char* bp_last_error(void);
int bp_version(void);

/* Create / destroy a context on CUDA device `device`.  Fails with BP_ERR_NO_DEVICE when there is no
 * sm_100 GPU: there is no CPU path. */
int bp_init(int device, bp_handle** out);
int bp_destroy(bp_handle* h);
/* Launch on the caller's CUDA stream (a cudaStream_t), e.g. torch's current stream. */
int bp_set_stream(bp_handle* h, void* cuda_stream);
int bp_synchronize(bp_handle* h);
/* Block the calling host thread until the intraday block of the last bp_upload_market_async has arrived in HBM (kernels
 * queued behind it may still be running).  Lets a caller that alternates between two handles start the upload of the
 * next market when the link is free instead of sharing it between two transfers (bench_configs.py, C5). */
int bp_wait_upload(bp_handle* h);
/* With enable != 0 the batched calls return as soon as their work is queued even when the outputs are HOST
 * buffers (which must then be page-locked): the results are complete after bp_synchronize().  Lets the host
 * plan the next batch (e.g. the conjugate windows) while the GPU still works on the previous one (Jeffreys).
 * Default 0: calls with host outputs return with the results in place. */
int bp_set_async_outputs(bp_handle* h, int enable);
/* Upper bound for the per-batch workspace (bytes); windows are processed in chunks that fit. */
int bp_set_workspace_limit(bp_handle* h, size_t bytes);
int bp_device_info(bp_handle* h, int* sm_count, size_t* free_bytes, size_t* total_bytes);
/* Number of kernels this handle has launched so far (bench.py's gpu_launches). */
long long bp_launch_count(bp_handle* h);

/* Per-stage device timing with CUDA events on the handle's stream.  bp_get_stage_times synchronises,
 * returns the summed milliseconds and launch counts per stage since the previous call, and resets. */
int bp_set_stage_timing(bp_handle* h, int enable);
int bp_get_stage_times(bp_handle* h, double* ms /*[BP_NSTAGE]*/, long long* launches /*[BP_NSTAGE]*/);

/* Work counters of the Gram stage since the previous call (then reset): out4[0] window rows contracted on
 * the tensor cores, [1] precomputed block tiles added, [2] rows contracted by the block precompute, [3] rows
 * a from-scratch contraction of every window would touch.  bench.py derives executed FLOPs / bytes from them. */
int bp_get_gram_work(bp_handle* h, double* out4);
/* Smallest batch (windows) for which the Gram kernel reuses precomputed block tiles between overlapping
 * windows; INT_MAX disables the reuse (every window is contracted from scratch). Default 32. */
int bp_set_reuse_min_windows(bp_handle* h, int min_windows);
/* Long intraday look-backs (the 252-day HF window of BASELINE config 3, reached in the reference through
 * conjugate_prior_S_df=, :299-318): the look-back of every window covers whole trading days, so the bars are cut into day
 * blocks at the hf_lo / hf_hi values of the batch, each block's Gram tile is contracted once, and for windows of at
 * least `min_days` blocks the tiles are scanned per chunk (suffix / prefix sums, no subtraction) so that a window adds
 * at most THREE stored tiles whatever its look-back; its column means come from the scanned per-day sums and S0 w0
 * from a by-product of the Gram launch, so no kernel walks the window's own rows.  0 disables (one tile per day).
 * Default 8. */
int bp_set_hf_presum_min_days(bp_handle* h, int min_days);
/* Jeffreys batches of CONSECUTIVE trade dates (calculate_mean_jeffreys_posterior_nu, :580-608): consecutive windows
 * differ by a rank 2k+4 term (k rows in, k rows out, the change of the risk-free adjustment and of t t'/n), so only
 * every `group`-th window is factorised and the others are solved relative to it by the Woodbury identity (30
 * triangular solves per group + a small elimination per window instead of a factorisation per window).  Each solved
 * window is held to an a-priori bound of the extended-precision solution (tests/_chain_ref.py).  group in [2, 8]; 0
 * or 1 factorises every window.  Default 8.  Batches that are not consecutive dates, weekly windows, and calls that
 * ask for T / S1 always take the per-window path. */
int bp_set_jeffreys_chain(bp_handle* h, int group);
/* Solve-stage work since the previous call (then reset): out2[0] windows factorised, out2[1] windows solved
 * relative to a base window. */
int bp_get_solve_work(bp_handle* h, double* out2);
/* enable != 0: every window the solver factorises also gets BP_SCAL_ANORM1 and BP_SCAL_RCOND (two more kernels per
 * solve launch, timed as BP_STAGE_COND), and the Jeffreys chain is not used (every window is factorised).  Weights,
 * nu, w1, status and scalar slots 0-9 are the same bits as with it off.  Default 0. */
int bp_set_condition_estimate(bp_handle* h, int enable);

/* Pipelining of bp_upload_market_async against bp_conjugate_batched: an intraday block of at least min_bytes
 * is copied in `segments` pieces (1..8; 1 disables; geometric: 1/2, 1/4, ... of the rows), and the conjugate
 * statistics / Gram stages of the windows whose bars have arrived run while the rest is still on the bus
 * (the per-date loop of the reference, main.py:74 -> portfolio_calculations.py:1127, has no such ordering
 * constraint: every date only reads bars up to that date).  Default: 8 segments from 256 MiB. */
int bp_set_upload_pipeline(bp_handle* h, int segments, long long min_bytes);
/* Explicit segment boundaries for the next asynchronous uploads: n cumulative row fractions (non-decreasing, the
 * last segment always ends at the last row); n = 0 restores the geometric default.  Once the kernels are faster than
 * the bus the best cut is one solver wave (bp_solve_wave_windows) of ready windows per segment with a short last
 * segment: every segment's windows are then solved at full occupancy while the next segment is on the bus, and only
 * the last few windows remain after the copy has finished. */
int bp_set_upload_fractions(bp_handle* h, int n, const double* cum_fractions);
/* Windows the solver works on concurrently (one CTA each, 6 per SM). */
int bp_solve_wave_windows(bp_handle* h);

/* Host -> HBM: replaces the pandas frames of get_market_data() (data_handling.py:270-291).  Also
 * computes both log-return matrices on the device (:37, :314). */
int bp_upload_market(bp_handle* h, const bp_market_desc* m);
/* Same, but returns as soon as the copies are queued: the host arrays must be page-locked and stay
 * valid until bp_synchronize().  The intraday block travels on a second stream, so a following
 * bp_jeffreys_batched / bp_stats_batched overlaps the transfer; conjugate calls wait for it. */
int bp_upload_market_async(bp_handle* h, const bp_market_desc* m);
/* Loop level (calculate_portfolio_weights, :954-988, slices the frames to the universe of EACH date; backtest_portfolio,
 * :1221-1238, does so once per trading day): the full market -- every candidate column, every row -- is uploaded ONCE
 * into a resident pool, and the working market of a batch (the universe of a run of dates in cap-descending order, the
 * rows its windows read) is gathered from it on the device: no host -> device transfer per asset set.
 * bp_upload_pool(h, NULL) releases the pool. */
int bp_upload_pool(bp_handle* h, const bp_market_desc* m);
typedef struct bp_pool_select {
    int n_cols;
    const int* cols;        /* pool columns, in the order they take in the working market */
    int day_lo, day_hi;     /* daily rows [day_lo, day_hi) of the pool */
    long long hf_lo, hf_hi; /* intraday rows [hf_lo, hf_hi) (equal: none) */
} bp_pool_select;
int bp_select_market(bp_handle* h, const bp_pool_select* s);
/* A STACKED working market: windows whose universes differ, evaluated in one batch.  Window w gets its own contiguous
 * block of rows -- daily pool rows [day_lo[w], day_hi[w]) (prices, caps, risk-free rate) and intraday pool rows
 * [hf_lo[w], hf_hi[w]) -- holding its own pool columns cols[w][0..n_cols), in that order.  The blocks follow one
 * another: block w starts at stack row day_off[w] (intraday: hf_off[w]), with day_off[0] = 0 and
 * day_off[w+1] = day_off[w] + day_hi[w] - day_lo[w] (the host's prefix sums; anything else is BP_ERR_INVALID, as is a
 * column or row range outside the pool).  A batch that follows names stack rows: a window must read its own block
 * only, which a block holding exactly the rows a bp_select_market slice would give that window guarantees (its rows
 * then sit at the same relative positions, and every kernel gives the same bits).
 * Windows of a stacked market share no rows, so the routes that share work between windows -- the Gram kernel's block
 * reuse and pre-summed day blocks, the banded daily pass, the Jeffreys chain -- are off for every batch on it, whatever
 * bp_set_reuse_min_windows / bp_set_jeffreys_chain say; the next bp_select_market / bp_upload_market restores them.
 * Weekly windows: bp_set_resampled then names rows of the stack (one set of shared weekly rows per window). */
typedef struct bp_window_select {
    int n_windows;                  /* W                                                                  */
    int n_cols;                     /* N: columns of every block                                          */
    const int* cols;                /* [W][N] pool columns of each window                                 */
    const int* day_lo;              /* [W] daily pool rows [day_lo, day_hi) of each block                 */
    const int* day_hi;
    const int* day_off;             /* [W] first stack row of each daily block                            */
    const long long* hf_lo;         /* [W] intraday pool rows [hf_lo, hf_hi) (equal: none); all three     */
    const long long* hf_hi;         /*     intraday arrays NULL: a stack without intraday rows           */
    const long long* hf_off;        /* [W] first stack row of each intraday block (< 2^31 rows in all)    */
} bp_window_select;
int bp_select_windows(bp_handle* h, const bp_window_select* s);
/* Re-run the log-return stage on the resident prices (device-only timing of the whole path). */
int bp_prepare_market(bp_handle* h);

/* calculate_canonical_statistics_t / _T (:163-245) for W windows. t:[W][N], T:[W][N][N]. */
int bp_stats_batched(bp_handle* h, const bp_window_batch* b, double* t, double* T);
/* calculate_conjugate_prior_n / _S (:247-267, :285-333): n0:[W], S0:[W][N][N] (= n0 * cov * m). */
int bp_hf_cov_batched(bp_handle* h, const bp_window_batch* b, double* n0, double* S0);
/* calculate_conjugate_hf_mcm_portfolio (:819-836) for W windows. */
int bp_conjugate_batched(bp_handle* h, const bp_window_batch* b, const bp_outputs* out);
/* calculate_jeffreys_portfolio (:838-849) for W windows. */
int bp_jeffreys_batched(bp_handle* h, const bp_window_batch* b, const bp_outputs* out);

/* Sibling estimators on the sample moments of the same daily window (SURVEY §8(f) rank 3); they share the
 * batched Gram and the batched Cholesky kernels of the Bayesian path.
 *  BP_ESTIMATOR_JORION     calculate_jorion_portfolio (:851-895): Bayes-Stein shrinkage of the sample mean towards
 *                          the grand mean mu_g and the matching predictive covariance V_PJ; ONE factorisation of the
 *                          centred Gram with two right-hand sides (t and 1), V_PJ^-1 by Sherman-Morrison.
 *                          Needs rolling_window - 1 > N + 2 (:879).  scalars: BP_SCAL_JORION_*.
 *  BP_ESTIMATOR_SHRINKAGE  calculate_shrinkage_portfolio (:703-758) in the closed form of the reference's own CHECK
 *                          (:748-756): weights = (1/gamma) Sigma_LW^-1 mu_hat with the Ledoit-Wolf covariance of
 *                          pypfopt's CovarianceShrinkage.ledoit_wolf() (= sklearn.covariance.ledoit_wolf).  The
 *                          reference returns these weights after a cvxpy solve and clean_weights() rounding; the
 *                          rounding is the Python shim's job.  scalars: BP_SCAL_LW_*.
 * Outputs honoured: weights, nu (weights before 1/gamma), w1 (C^-1 t), t, rhs, scalars, status, S1 (Jorion: the
 * centred Gram C = (m-1) V_hat; shrinkage: m Sigma_LW / (1 - s) with s the shrinkage intensity, and rhs = t / (1 - s)),
 * m = rolling_window - 1.  As in sklearn, s = 0 for one asset, and s = 1 exactly when beta >= delta (the intensity
 * clips): Sigma_LW = mu I, and then S1 = m Sigma_LW = mu m I and rhs = t. */
#define BP_ESTIMATOR_JORION 1
#define BP_ESTIMATOR_SHRINKAGE 2
#define BP_SCAL_JORION_MU_G 0          /* grand mean                                  :882               */
#define BP_SCAL_JORION_LAMBDA 1        /* lambda_hat                                  :885               */
#define BP_SCAL_JORION_V 2             /* v_hat                                       :887               */
#define BP_SCAL_JORION_Q 4             /* (mu_hat - mu_g 1)' V_bar^-1 (mu_hat - mu_g 1)                  */
#define BP_SCAL_JORION_ONE_VINV_ONE 5  /* 1' V_bar^-1 1                                                  */
#define BP_SCAL_LW_SHRINKAGE 0         /* Ledoit-Wolf shrinkage intensity                                */
#define BP_SCAL_LW_MU 1                /* trace(emp_cov) / N                                             */
#define BP_SCAL_LW_BETA 2
#define BP_SCAL_LW_DELTA 4
int bp_estimator_batched(bp_handle* h, const bp_window_batch* b, int estimator, const bp_outputs* out);

/* The posterior MOMENTS of W windows without the solve: any of t, w0, rhs, scalars (n0, n1, c, v0, MCM
 * average), T, S0, S1 (mode 0: conjugate S1 = S0 + T, :335-358; mode 1: Jeffreys T - tt'/n, :600-601).
 * Backs calculate_average_mcm_window / calculate_conjugate_prior_n / _posterior_n / _prior_w /
 * _posterior_S / calculate_conjugate_c when nothing is injected (:90-114, :247-430). */
int bp_moments_batched(bp_handle* h, const bp_window_batch* b, int mode, const bp_outputs* out);

/* Backtest loop body (:1054-1104, :1127-1219) for a whole backtest: daily portfolio simple returns with
 * weight drift between rebalances, turnover and transaction cost at each rebalance, weight metrics and
 * the distance to the value-weighted comparison portfolio.  The first rebalance date is the backtest
 * start (:1166-1167).  All pointers may be host or device. */
typedef struct {
    int n_rebalances;            /* R                                                                */
    const int* reb_row;          /* [R] daily rows of the rebalance dates, ascending (:1166-1176)     */
    int last_row;                /* daily row of ts_end_date (>= reb_row[R-1]); later days only drift  */
    const double* weights;       /* [R][N] weights chosen at each rebalance, uploaded column order,
                                    0 for stocks outside that date's universe                        */
    const unsigned char* member; /* [R][N] 1 = stock is in that date's universe; NULL = all stocks    */
    double distance_scale;       /* spec["risk_aversion"] or 1 (:1101)                               */
    double turnover_cost_bps;    /* spec["turnover_cost"] (:1214)                                    */
    double* returns;             /* [last_row - reb_row[0]]      portfolio_simple_returns_series      */
    double* turnover;            /* [R-1]                        portfolio_turnover_series           */
    double* metrics;             /* [R][5] max_long, max_short, avg_long, avg_short, average distance */
} bp_backtest_desc;
int bp_backtest_batched(bp_handle* h, const bp_backtest_desc* d);

/* performance_metrics (portfolio_evaluation.py:464-701) for an ENSEMBLE of return series at once (64 synthetic paths x
 * strategies): one row of BP_PM_COUNT statistics per series.  returns / excess: [n_paths][n_obs] HOST arrays (simple
 * returns after adjust_returns, :46-72, and excess returns, :703-719); years = (index[-1] - index[0]).days / 365 (:524);
 * out: [n_paths][BP_PM_COUNT] host.  The probabilistic Sharpe ratio (:78-120) follows on the host from BP_PM_SKEW,
 * BP_PM_KURT and BP_PM_SHARPE_1 of the series and of the benchmark.
 * BP_PM_SKEW and BP_PM_KURT are NaN for a flat excess series, by scipy.stats' rule m2 <= (DBL_EPSILON * mean)^2 on the
 * kernel's mean and the two-pass corrected m2 = (sum b^2 - (sum b)^2 / n) / n, b = excess - mean: the correction
 * cancels the rounding error of the mean, so a constant series is NaN even when its computed mean is a few ulp off.
 * The other statistics use the uncorrected m2 = sum b^2 / n. */
enum {
    BP_PM_CUM_RETURN = 0, BP_PM_CAGR, BP_PM_SHARPE, BP_PM_SORTINO, BP_PM_MAX_DD, BP_PM_CALMAR, BP_PM_AVG_LOSS,
    BP_PM_AVG_RETURN, BP_PM_AVG_WIN, BP_PM_BEST, BP_PM_WORST, BP_PM_ANN_VOL, BP_PM_DAILY_VAR, BP_PM_SKEW, BP_PM_KURT,
    BP_PM_SHARPE_1, BP_PM_COUNT
};
int bp_path_metrics(bp_handle* h, int n_paths, int n_obs, const double* returns, const double* excess, double years,
                    double* out);

/* calculate_excess_log_returns_from_prices (:31-62) of ONE window (b->n_windows == 1):
 * X is [(rolling_window-1)][N]. */
int bp_excess_returns(bp_handle* h, const bp_window_batch* b, double* X);

/* calculate_portfolio_variance (:64-88): *out = w' S w for dense S [n][n] (host pointers). */
int bp_quadratic_form(bp_handle* h, int n, const double* w, const double* S, double* out);

/* Single-window posterior from DENSE, possibly caller-injected moments: the optional-argument forms of
 * calculate_conjugate_c / _posterior_S / _posterior_w / calculate_mean_conjugate_posterior_nu (:382-577)
 * and calculate_mean_jeffreys_posterior_nu (:580-608).  All pointers are host pointers. */
typedef struct {
    int n_assets;
    int jeffreys;               /* 0 conjugate, 1 Jeffreys                                           */
    int rolling_window;         /* n                                                                 */
    double risk_aversion;
    const double* T;            /* [N][N] canonical statistic T; NULL (with t NULL): only v0 and c
                                   are computed (calculate_conjugate_c with injected moments)        */
    const double* t;            /* [N]                                                               */
    const double* S0;           /* [N][N] conjugate prior S        (conjugate only)                  */
    const double* w0;           /* [N]    prior weights            (conjugate only)                  */
    double n0;                  /* conjugate prior n                                                 */
    const double* n1;           /* optional injected posterior n   (NULL: n0 + n)                    */
    const double* c;            /* optional injected conjugate_c                                     */
    const double* S1;           /* optional injected posterior S [N][N]                              */
    const double* w1;           /* optional injected posterior w [N]                                 */
} bp_dense_problem;

typedef struct {
    double* scalars;            /* [BP_NSCAL] n0, n1, c, v0, v1                                       */
    double* S1;                 /* [N][N]                                                            */
    double* w1;                 /* [N]                                                               */
    double* nu;                 /* [N]                                                               */
    double* weights;            /* [N]                                                               */
    int* status;                /* [1]                                                               */
} bp_dense_result;

int bp_dense_posterior(bp_handle* h, const bp_dense_problem* in, const bp_dense_result* out);

/* The solve stage alone on caller-supplied matrices, W windows at once: the batched form of the injected-moment calls
 * calculate_conjugate_posterior_w / calculate_mean_conjugate_posterior_nu with conjugate_posterior_S_df= (:485-489,
 * :572-575), calculate_mean_jeffreys_posterior_nu (:600-606) and Jorion from C and t (:851-895).  No market is needed.
 * Outputs honoured: weights, nu, w1, scalars (v1 in BP_SCAL_V1, n1 in BP_SCAL_N1; Jorion: BP_SCAL_JORION_*) and
 * status; asking for T, S0, S1, t, w0 or rhs is an error.  The solver accepts N <= 3072 (Jorion: N <= 1536). */
typedef struct {
    int n_windows, n_assets;    /* W, N                                                              */
    int jeffreys;               /* 0: nu = (n1 + N + 2) w1 / (n1 - w1' S w1); 1: nu = w1             */
    int estimator;              /* 0, or BP_ESTIMATOR_JORION: S = C, rhs = t, and a right-hand side of
                                   ones rides along (jeffreys and n1 are then ignored)               */
    int n_returns;              /* Jorion's m, must exceed N + 2                                     */
    double risk_aversion;
    const double* S;            /* [W][N][N] host; only the lower triangle is read                   */
    const double* rhs;          /* [W][N] host                                                       */
    const double* n1;           /* [W] host, conjugate scaling only                                  */
} bp_solve_desc;
int bp_solve_batched(bp_handle* h, const bp_solve_desc* d, const bp_outputs* out);

#ifdef __cplusplus
}
#endif
#endif /* BAYES_PORTFOLIO_H */
