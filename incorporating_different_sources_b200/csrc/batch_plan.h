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
};

inline long long floor_div(long long a, long long b) { return a >= 0 ? a / b : -((-a + b - 1) / b); }

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
// Plans a batch that check_batch accepted.  Fails only when the plan is internally inconsistent.
int plan_batch(const PlanCtx& ctx, const bp_window_batch* b, bool need_hf, BatchPlan* plan, std::string* err);
// Writes the descriptor image (plan.ints ints) to dst.
void write_batch(const BatchPlan& plan, const bp_window_batch* b, int* dst);

}  // namespace bp
