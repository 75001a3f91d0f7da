// Host-side planning of a window batch: validation, the block grids of the Gram kernel's window-overlap reuse and the
// descriptor image the kernels read.  No CUDA runtime call and no kernel: the CPU tests compile batch_plan.cu alone.
#pragma once
#include <array>
#include <cstddef>
#include <map>
#include <string>
#include <utility>
#include <vector>

#include "../../include/bayes_portfolio.h"
#include "kernels.h"

namespace bp {

// what the planner reads from the handle
struct PlanCtx {
    bool has_market = false;
    int N = 0, ld = 0, D = 0, Rw = 0, n_mcm = 0;
    long long R = 0;
    long long hf_extra_rows = 0;       // rows behind the intraday returns for gathered overnight returns
    bool has_caps = false;
    bool has_mcm_w = false;            // bp_set_resampled was given MCM rows
    size_t ws_limit = 0;
    int reuse_min_windows = 32;
    int presum_min_days = 8;
    int stride = 1;                    // chain path: only every stride-th window goes through the Gram kernel
    bool stacked = false;              // stacked market (bp_select_windows): windows share no rows, no block reuse / band
    // stacked market: first stack row of every block (daily; intraday or nullptr) and the price rows of the resampled
    // rows (bp_set_resampled, or nullptr), so that each window of a batch is held to one block
    int n_blocks = 0;
    const long long* day_block = nullptr;
    const long long* hf_block = nullptr;
    const int* rs_num = nullptr;
    const int* rs_den = nullptr;
    // route choice (plan_chain_group, plan_route)
    bool cond_estimate = false;        // bp_set_condition_estimate: every window must be factorised
    int chain_group = 0;               // bp_set_jeffreys_chain
    int chain_max = 0;                 // chain_max_group()
    bool chain_smem_fits = false;      // chain_smem_bytes(N) <= 227 KB
    bool hf_pending = false;           // an asynchronous intraday upload is still in flight ...
    int n_seg = 0, seg_waited = 0;     // ... in n_seg segments, of which seg_waited have been waited for
};

// What a batched call computes: the route decisions depend on it
struct CallDesc {
    int mode = BP_MODE_CONJUGATE;
    bool solve = false;
    int estimator = BP_EST_NONE;
    bool T = false, S0 = false, S1 = false;        // these outputs are requested
};

inline long long floor_div(long long a, long long b) { return a >= 0 ? a / b : -((-a + b - 1) / b); }
inline int round_up(int x, int m) { return (x + m - 1) / m * m; }

// Workspace layout of one window: the solver matrix (ldS columns, rowsS rows) and the vectors (ldv doubles each)
struct Layout {
    int N, ldv, ldS, rowsS;
    long long win_stride, y_stride, mv_stride;
    size_t per_window;
};

// max_m: longest intraday window (scratch of the row dots); with_mv: room for the Gram kernel's G w0 partials
Layout make_layout(int N, int ld, int max_m, bool with_mv);

// Block grids of one phase, two levels (0 = coarse, 1 = fine; the fine size divides the coarse size): block b of
// level l covers return rows [b*blk[l], (b+1)*blk[l]); blk[l] == 0: level unused
struct PhasePlan {
    int blk[2] = {0, 0};
    int bmin[2] = {0, 0}, nb[2] = {0, 0};
    // "inner" day blocks: every hf_lo / hf_hi of the batch is a block boundary (the HF look-back always covers whole
    // days, :310-312, whatever the bar calendar), block b = return rows starts[b]+1 .. starts[b+1]-1, i.e. a trading
    // day WITHOUT its first (overnight) return; the overnight rows are gathered into a compact row range behind the
    // intraday matrix, so a window is [its days' inner blocks] + [one short run of overnight rows]
    bool inner = false;
    std::vector<int> starts;
    // pre-summed runs (long look-backs): chunk > 0 -> a window adds suffix'[first day] + prefix[...] tiles (<= 3)
    int chunk = 0;
};

typedef std::array<long long, 6> RunKey;       // (coarse, fineA, fineB) block runs [lo, hi) of a daily window

struct BatchPlan {
    int W = 0, n = 0, max_m = 0, mcm_rows = 0, stride = 1;
    long long R = 0;                   // first gathered overnight row
    bool need_hf = false, resampled = false;
    PhasePlan phase[2];                // 0 = intraday, 1 = daily
    bool presum = false;               // windows add <= 3 scanned tiles (PhasePlan::chunk)
    bool band_ok = false;              // consecutive trade dates: the daily pass runs as a banded GEMM
    // phase B (daily rows): each distinct run [lo, hi) of whole blocks is summed once (range_sum_kernel), and each
    // distinct (coarse, fine, fine) run triple of a window is combined once (combine_runs_kernel)
    std::map<std::pair<long long, long long>, int> range_id[2];
    std::map<RunKey, int> full_id;
    int nranges[2] = {0, 0}, nfull = 0;
    // descriptor image, offsets in ints: 7 columns [W] (day_row, span, row0, hf_row0, hf_span, extra_row, caps_row),
    // Gram jobs [W][GRAM_DESC_INTS], block jobs [phase][level][nb][GRAM_DESC_INTS], ranges [level][n][2],
    // triples [nfull][3], day-block starts [nb + 1] (inner), scanned-vector ids [W][3] (presum)
    size_t off_gram = 0, off_blocks[2][2] = {{0, 0}, {0, 0}}, off_ranges[2] = {0, 0}, off_triples = 0,
           off_starts = 0, off_vids = 0, ints = 0;
    // device stores the batch needs, in doubles
    size_t store[2][2] = {{0, 0}, {0, 0}}, rstore[2] = {0, 0}, fstore = 0, vstore = 0;
    // increments of the Gram-stage work counters (bp_get_gram_work)
    double work_k_rows = 0, work_add_blocks = 0, work_pre_rows = 0, work_full_rows = 0;
};

// Formats an error message into *err and returns code.
int fail_to(std::string* err, int code, const char* fmt, ...);
// Every validation of a batch against the resident market; BP_OK or a BP_ERR_* code with the message in *err.
int check_batch(const PlanCtx& ctx, const bp_window_batch* b, bool need_hf, std::string* err);
// The call's own arguments (risk aversion, Jorion's T - N - 2 > 0) for a batch check_batch accepted.
int check_call(const PlanCtx& ctx, const bp_window_batch* b, const CallDesc& call, std::string* err);
// Chain group G of a batch check_batch accepted: >= 2 factorises only every G-th window and solves the others
// relative to it (jeffreys_chain.cu); plan_batch takes it as its stride.
int plan_chain_group(const PlanCtx& ctx, const bp_window_batch* b, const CallDesc& call);
// Plans a batch that check_batch accepted.  Fails only when the plan is internally inconsistent.
int plan_batch(const PlanCtx& ctx, const bp_window_batch* b, bool need_hf, BatchPlan* plan, std::string* err);
// Writes the descriptor image (plan.ints ints) to dst.
void write_batch(const BatchPlan& plan, const bp_window_batch* b, int* dst);

// How the driver runs a planned batch
struct Route {
    int G = 0;                         // chain group (plan_chain_group)
    // prep + Gram of the windows whose intraday bars have arrived run between the segments of an asynchronous upload
    bool pipelined = false;
    int Wc = 0;                        // windows per workspace chunk
    long long hf_wait_rows = 0;        // > 0: wait for the intraday price rows below this before the batch
    Layout L{};
};
// Route of a batch plan_batch planned with stride G.  Fails only when the route is internally inconsistent.
int plan_route(const PlanCtx& ctx, const BatchPlan& plan, const bp_window_batch* b, const CallDesc& call, int G,
               Route* route, std::string* err);

}  // namespace bp
