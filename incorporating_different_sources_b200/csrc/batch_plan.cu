// Window-batch planning on the host (see batch_plan.h).  It decides which rows of every window are contracted on the
// tensor cores and which come from precomputed block tiles, hence the summation order of every Gram tile.
#include "batch_plan.h"

#include <algorithm>
#include <cstdarg>
#include <cstdio>
#include <cstring>

namespace bp {

int fail_to(std::string* err, int code, const char* fmt, ...) {
    char buf[1024];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof(buf), fmt, ap);
    va_end(ap);
    *err = buf;
    return code;
}

namespace {

// Split of the row range [row0, row0+rows) of a window: head rows, fine blocks, coarse blocks, fine blocks, tail rows
struct Split {
    long long k0_row = 0, k0_n = 0, k1_row = 0, k1_n = 0;     // rows contracted on the tensor cores
    long long c_lo = 0, c_hi = 0;                             // coarse blocks [c_lo, c_hi)
    long long fa_lo = 0, fa_hi = 0, fb_lo = 0, fb_hi = 0;     // fine blocks on the head / tail side
};

Split split_rows(int row0, int rows, const PhasePlan& P) {
    Split s;
    s.k0_row = row0;
    s.k0_n = rows;
    if (rows <= 0 || (P.blk[0] <= 0 && P.blk[1] <= 0)) return s;
    const long long r0 = row0, r1 = r0 + rows;
    long long head_end = r1, tail_begin = r1;      // head = [r0, head_end), tail = [tail_begin, r1)
    if (P.blk[0] > 0) {
        const long long B = P.blk[0];
        const long long lo = floor_div(r0 + B - 1, B), hi = floor_div(r1, B);
        if (hi > lo) {
            s.c_lo = lo;
            s.c_hi = hi;
            head_end = lo * B;
            tail_begin = hi * B;
        }
    }
    if (P.blk[1] > 0) {
        const long long F = P.blk[1];
        if (s.c_hi > s.c_lo) {
            const long long f_lo = floor_div(r0 + F - 1, F), f_hi = floor_div(r1, F);
            s.fa_lo = f_lo;  s.fa_hi = head_end / F;          // head_end is a multiple of the coarse (hence fine) size
            s.fb_lo = tail_begin / F;  s.fb_hi = f_hi;
            s.k0_n = f_lo * F - r0;
            s.k1_row = f_hi * F;
            s.k1_n = r1 - f_hi * F;
        } else {
            const long long f_lo = floor_div(r0 + F - 1, F), f_hi = floor_div(r1, F);
            if (f_hi > f_lo) {
                s.fa_lo = f_lo;  s.fa_hi = f_hi;
                s.k0_n = f_lo * F - r0;
                s.k1_row = f_hi * F;
                s.k1_n = r1 - f_hi * F;
            }
        }
    } else if (s.c_hi > s.c_lo) {
        s.k0_n = head_end - r0;
        s.k1_row = tail_begin;
        s.k1_n = r1 - tail_begin;
    }
    return s;
}

// split of window w's rows in phase ph; inner-block plans take every day of the window as a whole block
Split split_of(const PhasePlan& P, const bp_window_batch* b, int n, int ph, int w) {
    if (ph == 0 && P.inner) {
        Split sp;
        sp.c_lo = std::lower_bound(P.starts.begin(), P.starts.end(), b->hf_lo[w]) - P.starts.begin();
        sp.c_hi = std::lower_bound(P.starts.begin(), P.starts.end(), b->hf_hi[w]) - P.starts.begin();
        return sp;
    }
    if (ph == 0) return split_rows(b->hf_lo[w] + 1, b->hf_hi[w] - b->hf_lo[w] - 1, P);
    return split_rows(b->day_row[w] - n + 2, n - 1, P);
}

RunKey run_key(const Split& s) { return RunKey{s.c_lo, s.c_hi, s.fa_lo, s.fa_hi, s.fb_lo, s.fb_hi}; }

// descriptor ints of one phase (GRAM_PHASE_INTS) from a split, block indices relative to the stores
void write_phase_desc(const Split& s, const PhasePlan& P, int* d) {
    d[0] = (int)s.k0_row; d[1] = (int)s.k0_n; d[2] = (int)s.k1_row; d[3] = (int)s.k1_n;
    d[4] = (int)(s.c_lo - P.bmin[0]);  d[5] = (int)(s.c_hi - s.c_lo);
    d[6] = (int)(s.fa_lo - P.bmin[1]); d[7] = (int)(s.fa_hi - s.fa_lo);
    d[8] = (int)(s.fb_lo - P.bmin[1]); d[9] = (int)(s.fb_hi - s.fb_lo);
    if (d[5] == 0) d[4] = 0;
    if (d[7] == 0) d[6] = 0;
    if (d[9] == 0) d[8] = 0;
}

// Gram job descriptor of window w (GRAM_DESC_INTS ints) and, on the pre-summed path, its scanned-vector ids (vid may
// be null).  False when a pre-summed run would span more than three chunks, which the plan rules out.
bool gram_job(const BatchPlan& P, const bp_window_batch* b, int w, int* d, int* vid) {
    const int n = P.n, dr = b->day_row[w];
    std::fill(d, d + GRAM_DESC_INTS, 0);
    if (P.need_hf) {
        const PhasePlan& A = P.phase[0];
        int* dA = d;
        write_phase_desc(split_of(A, b, n, 0, w), A, dA);
        if (P.presum) {
            // suffix'[first day] (+ one whole chunk) (+ prefix[last day]): explicit tile ids into the unified store
            // [inner | suffix' | prefix]; the same ids address the scanned column sums (hf_vids)
            const int nb0 = A.nb[0], C = A.chunk, c_lo = dA[4], last = dA[4] + dA[5] - 1;
            const int qa = c_lo / C, s_next = std::min((qa + 1) * C, nb0);
            int ids[3] = {nb0 + c_lo, -1, -1};
            if (s_next <= last) {
                const int ql = last / C;
                if (ql > qa + 2) return false;
                if (ql == qa + 2) ids[1] = 2 * nb0 + (qa + 2) * C - 1;
                ids[2] = 2 * nb0 + last;
            }
            dA[0] = dA[1] = dA[2] = dA[3] = 0;
            for (int k = 0; k < 3; ++k) { dA[4 + 2 * k] = ids[k] >= 0 ? ids[k] : 0; dA[5 + 2 * k] = ids[k] >= 0 ? 1 : 0; }
            if (vid) std::copy(ids, ids + 3, vid);
        } else if (A.inner) {
            // overnight returns of days 2..last of the window: a run of dA[5]-1 gathered rows behind the matrix
            dA[0] = (int)(P.R + dA[4] + 1);
            dA[1] = dA[5] - 1;
        }
    }
    int* dB = d + GRAM_PHASE_INTS;
    if (P.resampled) {
        dB[0] = dr - (n - 2) + 1; dB[1] = n - 2;       // shared weekly rows
        dB[2] = b->extra_row[w];  dB[3] = 1;           // the trade date's own row
    } else if (w % P.stride == 0) {
        const Split sp = split_of(P.phase[1], b, n, 1, w);
        write_phase_desc(sp, P.phase[1], dB);
        // the whole-block runs of the window are combined into one tile per distinct (coarse, fine, fine) triple:
        // the coarse slot points into fstore
        if (dB[5] > 0 || dB[7] > 0 || dB[9] > 0) {
            dB[4] = P.full_id.at(run_key(sp));
            dB[5] = 1;
            dB[6] = dB[7] = dB[8] = dB[9] = 0;
        }
    }
    return true;
}

// Day blocks: the HF look-back of every window covers whole days, so the sorted set of all hf_lo / hf_hi values cuts
// the bars into blocks of which every window is a run -- whatever the bar calendar (half days, holidays).
std::vector<int> day_block_starts(const bp_window_batch* b) {
    const int W = b->n_windows;
    std::vector<int> st;
    st.reserve(2 * (size_t)W);
    for (int w = 0; w < W; ++w) { st.push_back(b->hf_lo[w]); st.push_back(b->hf_hi[w]); }
    std::sort(st.begin(), st.end());
    st.erase(std::unique(st.begin(), st.end()), st.end());
    if (st.size() < 3) return st;
    // stretches no window starts or ends in (the look-back of the first windows of a short batch) would be single
    // giant blocks contracted by one CTA per tile pair: cut them to the typical block length (a window contains such a
    // stretch entirely or not at all, so any cut inside it is a valid boundary)
    std::vector<int> gaps(st.size() - 1);
    for (size_t k = 0; k + 1 < st.size(); ++k) gaps[k] = st[k + 1] - st[k];
    std::nth_element(gaps.begin(), gaps.begin() + gaps.size() / 2, gaps.end());
    const int typical = std::max(8, gaps[gaps.size() / 2]);
    std::vector<int> cut;
    cut.reserve(st.size());
    for (size_t k = 0; k + 1 < st.size(); ++k) {
        cut.push_back(st[k]);
        const int gap = st[k + 1] - st[k];
        if (gap > 2 * typical) {
            const int pieces = gap / typical;
            for (int q = 1; q < pieces; ++q) cut.push_back(st[k] + (int)((long long)gap * q / pieces));
        }
    }
    cut.push_back(st.back());
    return cut;
}

}  // namespace

int check_batch(const PlanCtx& ctx, const bp_window_batch* b, bool need_hf, std::string* err) {
    if (!ctx.has_market) return fail_to(err, BP_ERR_STATE, "no market uploaded: call bp_upload_market first");
    const int W = b->n_windows, n = b->rolling_window;
    if (W <= 0) return fail_to(err, BP_ERR_INVALID, "n_windows must be positive");
    if (n < 3) return fail_to(err, BP_ERR_INVALID, "rolling_window must be >= 3");
    if (!b->day_row || !b->span_days) return fail_to(err, BP_ERR_INVALID, "day_row / span_days missing");
    if (need_hf) {
        if (!b->hf_lo || !b->hf_hi) return fail_to(err, BP_ERR_INVALID, "hf_lo / hf_hi missing");
        if (ctx.R <= 0) return fail_to(err, BP_ERR_STATE, "the uploaded market has no intraday prices");
        if (b->resampled && !b->prior_n && !ctx.has_mcm_w) return fail_to(err, BP_ERR_STATE, "bp_set_resampled was given no MCM rows");
        if (!b->prior_n && (b->mcm_index < 0 || b->mcm_index >= ctx.n_mcm))
            return fail_to(err, BP_ERR_INVALID, "mcm_index %d out of range", b->mcm_index);
        if (b->mcm_rows < 0 || b->mcm_rows > n) return fail_to(err, BP_ERR_INVALID, "mcm_rows must be in [0, rolling_window]");
        if (b->prior_weights == 0 && !ctx.has_caps) return fail_to(err, BP_ERR_STATE, "value-weighted prior needs market caps");
    }
    const bool rs = b->resampled != 0;
    if (rs) {
        if (ctx.Rw <= 0) return fail_to(err, BP_ERR_STATE, "resampled windows need bp_set_resampled first");
        if (!b->extra_row || !b->caps_row) return fail_to(err, BP_ERR_INVALID, "resampled windows need extra_row and caps_row");
    }
    for (int w = 0; w < W; ++w) {
        const int dr = b->day_row[w];
        if (rs) {
            // shared weekly rows dr-(n-2)+1 .. dr (row 0 is the zero row of the first week) + one per-date row
            if (dr - (n - 2) + 1 < 1 || dr >= ctx.Rw)
                return fail_to(err, BP_ERR_INVALID, "window %d: resampled day_row %d needs %d prior rows inside [1,%d)", w, dr, n - 2, ctx.Rw);
            if (b->extra_row[w] < 0 || b->extra_row[w] >= ctx.Rw || b->caps_row[w] < 0 || b->caps_row[w] >= ctx.D)
                return fail_to(err, BP_ERR_INVALID, "window %d: extra_row / caps_row out of range", w);
        } else if (dr < n - 1 || dr >= ctx.D) {
            return fail_to(err, BP_ERR_INVALID, "window %d: day_row %d needs %d prior price rows inside [0,%d)", w, dr, n - 1, ctx.D);
        }
        if (need_hf && !b->prior_n && dr < (b->mcm_rows ? b->mcm_rows : n) - 1 - (rs ? 1 : 0))
            return fail_to(err, BP_ERR_INVALID, "window %d: not enough MCM observations before day_row %d", w, dr);
        if (b->span_days[w] <= 0) return fail_to(err, BP_ERR_INVALID, "window %d: span_days must be positive", w);
        if (need_hf) {
            const int lo = b->hf_lo[w], hi = b->hf_hi[w];
            const int m = hi - lo - 1;
            if (lo < 0 || (long long)hi > ctx.R || m < 2)
                return fail_to(err, BP_ERR_INVALID, "window %d: intraday rows [%d,%d) give %d returns (need >= 2, rows < %lld)", w, lo, hi, m, ctx.R);
        }
    }
    if (ctx.n_blocks > 0) {
        // stacked market: every row a window reads (prices, caps, resampled rows' prices, intraday bars) lies in ONE
        // window's block, the same block for the daily and the intraday rows
        auto block_of = [&ctx](const long long* start, long long row) {
            return (int)(std::upper_bound(start, start + ctx.n_blocks, row) - start) - 1;
        };
        for (int w = 0; w < W; ++w) {
            const int dr = b->day_row[w];
            int blk;
            bool ok = true;
            if (rs) {
                blk = block_of(ctx.day_block, b->caps_row[w]);
                ok = ctx.rs_num && ctx.rs_den;
                for (int i = dr - (n - 2) + 1; ok && i <= dr + 1; ++i) {
                    const int row = i <= dr ? i : b->extra_row[w];
                    ok = block_of(ctx.day_block, ctx.rs_num[row]) == blk && block_of(ctx.day_block, ctx.rs_den[row]) == blk;
                }
            } else {
                blk = block_of(ctx.day_block, dr - n + 1);
                ok = block_of(ctx.day_block, dr) == blk;
            }
            if (ok && need_hf)
                ok = ctx.hf_block && block_of(ctx.hf_block, b->hf_lo[w]) == blk && block_of(ctx.hf_block, b->hf_hi[w] - 1) == blk;
            if (!ok)
                return fail_to(err, BP_ERR_INVALID, "window %d reads stack rows outside one window's block (bp_select_windows)", w);
        }
    }
    return BP_OK;
}

int check_call(const PlanCtx& ctx, const bp_window_batch* b, const CallDesc& call, std::string* err) {
    if (call.solve && (call.mode == BP_MODE_CONJUGATE || call.estimator != BP_EST_NONE) && !(b->risk_aversion != 0.0))
        return fail_to(err, BP_ERR_INVALID, "risk_aversion must be non-zero");
    if (call.estimator == BP_EST_JORION && b->rolling_window - 1 - ctx.N - 2 <= 0)
        return fail_to(err, BP_ERR_INVALID, "Jorion needs T - N - 2 > 0 (T = rolling_window - 1 returns, :879)");
    return BP_OK;
}

Layout make_layout(int N, int ld, int max_m, bool with_mv) {
    Layout L;
    L.N = N;
    L.ldv = ld;
    L.ldS = round_up(N, 32);
    L.rowsS = L.ldS + 8;
    L.win_stride = (long long)L.rowsS * L.ldS;
    L.y_stride = round_up(std::max(max_m, 2), 2);
    const int nt = (N + GRAM_TILE - 1) / GRAM_TILE;
    L.mv_stride = with_mv ? (long long)(nt * (nt + 1) / 2) * 2 * GRAM_TILE : 0;
    L.per_window = sizeof(double) * ((size_t)L.win_stride + 9 * (size_t)L.ldv + BP_NSCAL + (size_t)L.y_stride + (size_t)L.mv_stride) + 16;
    return L;
}

int plan_chain_group(const PlanCtx& ctx, const bp_window_batch* b, const CallDesc& call) {
    // Jeffreys batches of consecutive trade dates.  Not with the condition estimate on: a chained window's matrix is
    // never factorised, so there is no factor to estimate from.
    if (ctx.cond_estimate || call.mode != BP_MODE_JEFFREYS || (call.estimator != BP_EST_NONE && call.estimator != BP_EST_JORION) ||
        !call.solve || call.T || call.S0 || call.S1 || b->resampled || ctx.stacked || ctx.chain_group < 2 ||
        b->n_windows < 2 * ctx.chain_group || !ctx.chain_smem_fits)
        return 0;
    for (int w = 1; w < b->n_windows; ++w)
        if (b->day_row[w] != b->day_row[0] + w) return 0;
    // the whole batch in one workspace chunk: the descriptors are planned for the base windows only
    if ((size_t)b->n_windows * make_layout(ctx.N, ctx.ld, 0, false).per_window > ctx.ws_limit) return 0;
    const int G = std::min(ctx.chain_group, ctx.chain_max);
    // Conditioning guard: window b+k is the base with k rows removed and k rows added; the down-dated matrix
    // has rank n-1-k, and its Woodbury pivots -1 + l'J_b^-1 l tend to 0 as n-1-k approaches N (leverage 1),
    // where the small system loses digits while no pivot is exactly zero.  Chain only with a margin of rows;
    // closer to the rank limit every window is factorised on its own (the path the parity tests pin).
    if (G >= 2 && b->rolling_window - 1 < ctx.N + 2 * G + 8) return 0;
    return G;
}

int plan_route(const PlanCtx& ctx, const BatchPlan& P, const bp_window_batch* b, const CallDesc& call, int G, Route* out,
               std::string* err) {
    Route& r = *out;
    r = Route();
    r.G = G;
    r.L = make_layout(ctx.N, ctx.ld, P.presum ? 0 : P.max_m, P.presum);
    r.Wc = (int)std::min<size_t>((size_t)P.W, std::max<size_t>(1, ctx.ws_limit / r.L.per_window));
    // (plan_chain_group checks the same layout for a chained batch, so this cannot trigger unless the two are changed
    // apart)
    if (r.Wc < P.W && G >= 2) return fail_to(err, BP_ERR_STATE, "internal: chained batch does not fit one workspace chunk");
    // Pipelined against a segmented asynchronous intraday upload: prep + Gram of the windows whose bars have
    // arrived run while the rest is still being copied; the solve follows for all windows at once.
    r.pipelined = call.mode == BP_MODE_CONJUGATE && ctx.hf_pending && ctx.n_seg > 1 && ctx.seg_waited < ctx.n_seg &&
                  call.solve && !call.T && !call.S0 && r.Wc >= P.W && !P.presum;
    if (call.mode == BP_MODE_CONJUGATE && !r.pipelined)
        for (int w = 0; w < P.W; ++w) r.hf_wait_rows = std::max<long long>(r.hf_wait_rows, b->hf_hi[w]);
    return BP_OK;
}

int plan_batch(const PlanCtx& ctx, const bp_window_batch* b, bool need_hf, BatchPlan* out, std::string* err) {
    BatchPlan& P = *out;
    P = BatchPlan();
    const int W = b->n_windows, n = b->rolling_window;
    const bool rs = b->resampled != 0;
    P.W = W;
    P.n = n;
    P.mcm_rows = b->mcm_rows ? b->mcm_rows : n;
    P.stride = ctx.stride;
    P.R = ctx.R;
    P.need_hf = need_hf;
    P.resampled = rs;
    PhasePlan* plan = P.phase;
    // ---- block grids for the window-overlap reuse of the Gram kernel
    const int npairs_t = ((ctx.N + GRAM_TILE - 1) / GRAM_TILE) * ((ctx.N + GRAM_TILE - 1) / GRAM_TILE + 1) / 2;
    const size_t tiles = (size_t)npairs_t * GRAM_BLOCK_TILE_DOUBLES;      // doubles per block
    if (W >= ctx.reuse_min_windows && !ctx.stacked) {
        const int K = n - 1;
        if (!rs) {          // resampled windows: shared weekly rows + one per-date row, no block reuse
            // Block sizes were tuned on the bench workload (N = 500): coarse/fine 128/32 for the 1007-row Jeffreys
            // window and 64/16 for the 251-row conjugate window gave 18.6 ms for the Gram stage, 512/64 + 128/32
            // 19.4 ms, a single level (128 / 64) 21.9 ms; neither the DMMA pipe (40-50 %) nor L2 (26-32 %) is
            // saturated then, the stage is bound by per-item latencies.
            if (K >= 512) { plan[1].blk[0] = 128; plan[1].blk[1] = 32; }
            else if (K >= 128) { plan[1].blk[0] = 64; plan[1].blk[1] = 16; }
        }
        if (need_hf) {
            // day blocks are worth it when the windows overlap (each block serves >= 2 windows on average)
            std::vector<int> st = day_block_starts(b);
            const long long nb = (long long)st.size() - 1;
            long long sumD = 0;
            int minD = 1 << 30, maxD = 0, min_rows = 1 << 30;
            for (int w = 0; w < W; ++w) {
                const int D = (int)(std::lower_bound(st.begin(), st.end(), b->hf_hi[w]) - std::lower_bound(st.begin(), st.end(), b->hf_lo[w]));
                sumD += D; minD = std::min(minD, D); maxD = std::max(maxD, D);
            }
            for (long long k = 0; k < nb; ++k) min_rows = std::min(min_rows, st[k + 1] - st[k]);
            if (nb >= 2 && minD >= 2 && min_rows >= 8 && sumD >= 2 * nb && nb <= ctx.hf_extra_rows) {
                plan[0].inner = true;
                plan[0].starts.swap(st);
                plan[0].blk[0] = 1;                 // level 0 in use (block sizes vary: see starts)
                const int minL = minD - 1, maxL = maxD - 1;       // full days (overnight return included) per window
                if (ctx.presum_min_days > 0 && minD >= ctx.presum_min_days && maxL <= 2 * minL &&
                    3 * (size_t)nb * tiles * sizeof(double) <= ctx.ws_limit)
                    plan[0].chunk = minL;
            } else if (b->hf_hi[0] - b->hf_lo[0] >= 3 * 64) {
                plan[0].blk[0] = 64;
                plan[0].blk[1] = 16;
            }
        }
    }
    // block ranges touched by the (Gram-stage) windows, per phase and level, and the distinct daily runs
    for (int ph = 0; ph < 2; ++ph) {
        if (plan[ph].blk[0] <= 0 && plan[ph].blk[1] <= 0) continue;
        long long lo[2] = {1LL << 40, 1LL << 40}, hi[2] = {-(1LL << 40), -(1LL << 40)};
        for (int w = 0; w < W; w += P.stride) {
            const Split sp = split_of(plan[ph], b, n, ph, w);
            if (sp.c_hi > sp.c_lo) { lo[0] = std::min(lo[0], sp.c_lo); hi[0] = std::max(hi[0], sp.c_hi); }
            if (sp.fa_hi > sp.fa_lo) { lo[1] = std::min(lo[1], sp.fa_lo); hi[1] = std::max(hi[1], sp.fa_hi); }
            if (sp.fb_hi > sp.fb_lo) { lo[1] = std::min(lo[1], sp.fb_lo); hi[1] = std::max(hi[1], sp.fb_hi); }
            if (ph == 1) {
                if (sp.c_hi > sp.c_lo) P.range_id[0].emplace(std::make_pair(sp.c_lo, sp.c_hi), 0);
                if (sp.fa_hi > sp.fa_lo) P.range_id[1].emplace(std::make_pair(sp.fa_lo, sp.fa_hi), 0);
                if (sp.fb_hi > sp.fb_lo) P.range_id[1].emplace(std::make_pair(sp.fb_lo, sp.fb_hi), 0);
                if (sp.c_hi > sp.c_lo || sp.fa_hi > sp.fa_lo || sp.fb_hi > sp.fb_lo) P.full_id.emplace(run_key(sp), 0);
            }
        }
        for (int l = 0; l < 2; ++l) {
            if (hi[l] <= lo[l]) { plan[ph].blk[l] = 0; plan[ph].nb[l] = 0; continue; }
            plan[ph].bmin[l] = (int)lo[l];
            plan[ph].nb[l] = (int)(hi[l] - lo[l]);
            if ((size_t)plan[ph].nb[l] * tiles * sizeof(double) > ctx.ws_limit / 2) {      // too big: give up the reuse of this phase
                plan[ph] = PhasePlan();
                P.store[ph][0] = P.store[ph][1] = 0;
                break;
            }
            // + suffix' and prefix tiles of every block on the pre-summed path
            P.store[ph][l] = (size_t)plan[ph].nb[l] * tiles * (ph == 0 && l == 0 && plan[0].chunk > 0 ? 3 : 1);
        }
    }
    if (plan[0].inner && plan[0].nb[0] != (int)plan[0].starts.size() - 1)
        return fail_to(err, BP_ERR_STATE, "internal: day-block plan out of step with its boundaries");
    P.presum = plan[0].inner && plan[0].chunk > 0;
    const int nb0 = plan[0].inner ? plan[0].nb[0] : 0;
    if (P.presum) P.vstore = 3 * (size_t)nb0 * ctx.ld;
    for (int l = 0; l < 2; ++l) {
        if (plan[1].blk[l] <= 0) P.range_id[l].clear();
        for (auto& kv : P.range_id[l]) kv.second = P.nranges[l]++;
        P.rstore[l] = (size_t)P.nranges[l] * tiles;
    }
    if (plan[1].blk[0] <= 0 && plan[1].blk[1] <= 0) P.full_id.clear();
    for (auto& kv : P.full_id) kv.second = P.nfull++;
    P.fstore = (size_t)P.nfull * tiles;
    // sections of the descriptor image, in order; the 7 columns come first
    auto section = [&P](size_t ints) {
        const size_t off = P.ints;
        P.ints += ints;
        return off;
    };
    section((size_t)7 * W);
    P.off_gram = section((size_t)GRAM_DESC_INTS * W);
    for (int ph = 0; ph < 2; ++ph)
        for (int l = 0; l < 2; ++l) P.off_blocks[ph][l] = section((size_t)GRAM_DESC_INTS * plan[ph].nb[l]);
    for (int l = 0; l < 2; ++l) P.off_ranges[l] = section(2 * (size_t)P.nranges[l]);
    P.off_triples = section(3 * (size_t)P.nfull);
    P.off_starts = section(plan[0].inner ? (size_t)nb0 + 1 : 0);
    P.off_vids = section(P.presum ? 3 * (size_t)W : 0);
    // work counters: rows on the tensor cores and block tiles added by the Gram stage, rows of a from-scratch pass
    auto r8 = [](int r) { return (r + 7) / 8 * 8; };
    int d[GRAM_DESC_INTS];
    for (int w = 0; w < W; ++w) {
        if (need_hf) P.max_m = std::max(P.max_m, b->hf_hi[w] - b->hf_lo[w] - 1);
        P.work_full_rows += (need_hf ? b->hf_hi[w] - b->hf_lo[w] - 1 : 0) + (n - 1);
        if (w % P.stride != 0) continue;
        if (!gram_job(P, b, w, d, nullptr))
            return fail_to(err, BP_ERR_STATE, "internal: pre-summed run spans more than three chunks");
        for (int ph = 0; ph < 2; ++ph) {
            const int* dp = d + ph * GRAM_PHASE_INTS;
            P.work_k_rows += r8(dp[1]) + r8(dp[3]);
            P.work_add_blocks += dp[5] + dp[7] + dp[9];
        }
    }
    for (int ph = 0; ph < 2; ++ph)
        for (int l = 0; l < 2; ++l) {
            if (ph == 0 && l == 0 && plan[0].inner) {
                for (int k = 0; k < nb0; ++k) P.work_pre_rows += r8(plan[0].starts[k + 1] - plan[0].starts[k] - 1);
                continue;
            }
            P.work_pre_rows += (double)plan[ph].nb[l] * r8(plan[ph].blk[l]);
        }
    // banded-GEMM daily pass: worth it when 32 consecutive windows share almost all of their rows
    bool ok = !rs && !ctx.stacked && W >= 32 && n >= 16;
    for (int w = 1; ok && w < W; ++w) ok = b->day_row[w] >= b->day_row[w - 1];
    P.band_ok = ok && (long long)b->day_row[W - 1] - b->day_row[0] <= 2LL * W;
    return BP_OK;
}

void write_batch(const BatchPlan& P, const bp_window_batch* b, int* dst) {
    const int W = P.W, n = P.n;
    memset(dst, 0, sizeof(int) * P.ints);
    for (int w = 0; w < W; ++w) {
        const int dr = b->day_row[w];
        dst[w] = dr;
        dst[(size_t)W + w] = b->span_days[w];
        dst[(size_t)2 * W + w] = P.resampled ? dr - (n - 2) + 1 : dr - n + 2;   // first RETURN row (F2: n prices -> n-1 returns)
        if (P.need_hf) {
            dst[(size_t)3 * W + w] = b->hf_lo[w] + 1;       // first HF return row: the window's first bar has no return (F5)
            dst[(size_t)4 * W + w] = b->hf_hi[w] - b->hf_lo[w] - 1;   // span; the prep kernel counts the kept rows m in it
        }
        dst[(size_t)5 * W + w] = P.resampled ? b->extra_row[w] : -1;
        dst[(size_t)6 * W + w] = P.resampled ? b->caps_row[w] : dr;
        gram_job(P, b, w, dst + P.off_gram + (size_t)w * GRAM_DESC_INTS, P.presum ? dst + P.off_vids + 3 * (size_t)w : nullptr);
    }
    // block precompute launches: one pseudo-window per block, rows of that block only
    for (int ph = 0; ph < 2; ++ph)
        for (int l = 0; l < 2; ++l) {
            const PhasePlan& pp = P.phase[ph];
            for (int k = 0; k < pp.nb[l]; ++k) {
                int* d = dst + P.off_blocks[ph][l] + (size_t)k * GRAM_DESC_INTS + GRAM_PHASE_INTS * ph;
                if (pp.inner) {           // the day without its overnight return
                    d[0] = pp.starts[k] + 1;
                    d[1] = pp.starts[k + 1] - pp.starts[k] - 1;
                } else {
                    d[0] = (pp.bmin[l] + k) * pp.blk[l];
                    d[1] = pp.blk[l];
                }
            }
        }
    // block runs to pre-sum (store-relative block indices)
    for (int l = 0; l < 2; ++l)
        for (const auto& kv : P.range_id[l]) {
            int* d = dst + P.off_ranges[l] + 2 * (size_t)kv.second;
            d[0] = (int)(kv.first.first - P.phase[1].bmin[l]);
            d[1] = (int)(kv.first.second - P.phase[1].bmin[l]);
        }
    for (const auto& kv : P.full_id) {
        const RunKey& k = kv.first;
        int* d = dst + P.off_triples + 3 * (size_t)kv.second;
        d[0] = k[1] > k[0] ? P.range_id[0].at(std::make_pair(k[0], k[1])) : -1;
        d[1] = k[3] > k[2] ? P.range_id[1].at(std::make_pair(k[2], k[3])) : -1;
        d[2] = k[5] > k[4] ? P.range_id[1].at(std::make_pair(k[4], k[5])) : -1;
    }
    if (P.phase[0].inner) std::copy(P.phase[0].starts.begin(), P.phase[0].starts.end(), dst + P.off_starts);
}

}  // namespace bp
