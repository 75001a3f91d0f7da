// C-ABI of libbayes_portfolio.so: market residency, window batches, stage orchestration.
// Declarations and the reference interfaces each entry point replaces: include/bayes_portfolio.h.
#include <cuda.h>
#include <cudaTypedefs.h>
#include <cuda_runtime.h>

#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstring>
#include <string>
#include <vector>

#include "../../include/bayes_portfolio.h"
#include "batch_plan.h"
#include "kernels.h"

using namespace bp;

static_assert(BP_NSCAL == bp::BP_S_COUNT, "scalar record size mismatch between header and kernels");

namespace {

thread_local std::string g_err;      // bp_last_error

#define fail(...) fail_to(&g_err, __VA_ARGS__)

#define CU_TRY(expr)                                                                                     \
    do {                                                                                                 \
        cudaError_t _e = (expr);                                                                         \
        if (_e != cudaSuccess)                                                                           \
            return fail(BP_ERR_CUDA, "%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e), __FILE__, __LINE__); \
    } while (0)

bool is_device_ptr(const void* p) {
    cudaPointerAttributes a;
    if (cudaPointerGetAttributes(&a, p) != cudaSuccess) {
        cudaGetLastError();
        return false;
    }
    return a.type == cudaMemoryTypeDevice || a.type == cudaMemoryTypeManaged;
}

// A grow-only buffer of `cap` elements: device memory, or page-locked host memory when `pinned` (see grow)
template <class T>
struct DevBuf {
    T* p = nullptr;
    size_t cap = 0;
    bool pinned = false;
};

template <class T>
void free_buf(DevBuf<T>& b) {
    if (b.pinned) cudaFreeHost(b.p);
    else cudaFree(b.p);
    b.p = nullptr;
    b.cap = 0;
}

}  // namespace

struct bp_handle {
    int device = 0;
    cudaStream_t stream = nullptr;
    int sm_count = 0;
    size_t ws_limit = (size_t)24 << 30;
    long long launches = 0;
    // market
    bool has_market = false;
    int N = 0, D = 0, ld = 0, n_mcm = 0;
    long long R = 0;
    // prices / caps / hf_prices keep the caller's dense [rows][N] layout; lr_d / lr_hf are padded to ld
    double *prices = nullptr, *lr_d = nullptr, *caps = nullptr, *hf_prices = nullptr, *lr_hf = nullptr,
           *mcm = nullptr, *rf_row = nullptr;
    bool has_caps = false;
    // resident POOL: the full market (every column, every row) kept in HBM so that the working market of a batch
    // (a column subset in a given order, a row range) is gathered on the device instead of uploaded again
    double *pool_prices = nullptr, *pool_caps = nullptr, *pool_hf = nullptr, *pool_rf = nullptr;
    int pool_N = 0, pool_D = 0;
    long long pool_R = 0;
    DevBuf<int> pool_cols;
    // stacked working market (bp_select_windows): one block of rows per window, no rows shared between windows, so no
    // route that shares work between windows may run; the per-window (first pool row, first stack row, rows) table
    bool stacked = false;
    DevBuf<long long> stack_rows;
    std::vector<long long> stack_day_start, stack_hf_start;     // first stack row of each block (check_batch)
    std::vector<int> rs_num_host, rs_den_host;                  // stacked market: price rows of the resampled rows
    // resampled (weekly) return rows: see bp_set_resampled
    double *lr_w = nullptr, *rf_w = nullptr, *mcm_w = nullptr;
    int* rs_idx = nullptr;
    int Rw = 0;
    CUtensorMap map_w;
    size_t cap_daily = 0, cap_hf = 0, cap_mcm = 0, cap_days = 0;   // allocated sizes (elements) for buffer reuse
    cudaStream_t copy_stream = nullptr;                  // intraday H2D + its log-return kernel
    cudaEvent_t ev_main = nullptr, ev_hf = nullptr;
    bool hf_pending = false;
    // an asynchronous intraday upload is cut into segments (copy + log returns + event each) so that the
    // conjugate stages of the early rebalance dates run while the later bars are still on the bus
    static constexpr int MAX_SEG = 8;
    int pipe_segments = MAX_SEG;
    size_t pipe_min_bytes = (size_t)256 << 20;
    int n_seg = 0, seg_waited = 0;
    int n_frac = 0;                            // > 0: explicit cumulative row fractions of the segments (bp_set_upload_fractions)
    double frac[MAX_SEG] = {0};
    long long lr_hf_done = 0;                  // intraday return rows < lr_hf_done have been computed
    DevBuf<unsigned char> hf_keep;             // [R] 1 = intraday return row kept, 0 = dropped (hf_returns)
    long long hf_extra_rows = 0;               // rows allocated behind lr_hf for gathered overnight returns
    int lr_hf_ld_cap = 1;
    long long lr_hf_rows_cap = 0;              // rows allocated for lr_hf (at the leading dimension it was allocated with)
    long long seg_end[MAX_SEG] = {0};          // return rows < seg_end[s] are valid once ev_seg[s] has fired
    cudaEvent_t ev_seg[MAX_SEG] = {nullptr};
    CUtensorMap map_d, map_hf;
    // descriptor images (batch_plan.h) on the device and their page-locked staging (read zero-copy by a kernel), in
    // two slots used alternately: planning the next batch on the host never waits for the GPU to have fetched (or
    // finished using) the previous one, only for the batch before that
    DevBuf<int> desc_slot[2];
    DevBuf<int> desc_host_slot[2] = {{nullptr, 0, true}, {nullptr, 0, true}};
    cudaEvent_t ev_desc[2] = {nullptr, nullptr};
    bool ev_desc_armed[2] = {false, false};
    int desc_turn = 0;
    bool async_outputs = false;        // host outputs are complete only after bp_synchronize (see bp_set_async_outputs)
    // block tile stores of the Gram kernel (window-overlap reuse) and the smallest batch that uses them
    DevBuf<double> store[2][2];        // [phase][level]
    DevBuf<double> rstore[2];          // phase-B range-sum stores [level]
    DevBuf<double> fstore;             // phase-B combined runs (coarse + fine + fine)
    int reuse_min_windows = 32;
    // pre-summed intraday day blocks (long HF look-backs): windows with at least this many trading days add <= 3 scanned
    // tiles instead of one tile per day (0 disables); vector store [3 nb][ld] of the scanned per-day column sums
    int presum_min_days = 8;
    DevBuf<double> vstore;
    // work counters of the Gram stage since the last bp_get_gram_work (bench.py's roofline accounting)
    double work_k_rows = 0, work_add_blocks = 0, work_pre_rows = 0, work_full_rows = 0;
    // Jeffreys windows of consecutive trade dates: only every chain_group-th window is factorised, the others are
    // solved relative to it (jeffreys_chain.cu); < 2 disables.  Work counters for bench.py's roofline accounting.
    int chain_group = 8;
    double work_factored = 0, work_chained = 0;
    // reciprocal condition estimate of every factorised window (bp_set_condition_estimate)
    bool cond_estimate = false;
    DevBuf<double> prior_n;
    // banded-GEMM daily pass (band_prep.cu): risk-free weights [W][band_ld] and their sums [W][2]
    DevBuf<double> band_aw, band_stats;
    // workspace
    DevBuf<unsigned char> ws, stage;
    bool need_sync = false;
    PFN_cuTensorMapEncodeTiled_v12000 encode = nullptr;
    // optional per-stage CUDA-event timing (bench.py's roofline numbers)
    bool timing = false;
    std::vector<cudaEvent_t> ev_pool;
    size_t ev_used = 0;
    struct Span { int stage; cudaEvent_t a, b; };
    std::vector<Span> spans;
    cudaEvent_t ev_t0 = nullptr;       // start of the last upload (BP_TIMELINE=1: spans are printed relative to it)
    bool t0_armed = false;
};

namespace {
struct StageTimer {
    bp_handle* h;
    int stage;
    cudaEvent_t a = nullptr, b = nullptr;
    StageTimer(bp_handle* h_, int stage_) : h(h_), stage(stage_) {
        if (!h->timing) return;
        while (h->ev_pool.size() < h->ev_used + 2) {
            cudaEvent_t e;
            if (cudaEventCreate(&e) != cudaSuccess) return;
            h->ev_pool.push_back(e);
        }
        a = h->ev_pool[h->ev_used++];
        b = h->ev_pool[h->ev_used++];
        cudaEventRecord(a, h->stream);
    }
    ~StageTimer() {
        if (!a) return;
        cudaEventRecord(b, h->stream);
        h->spans.push_back({stage, a, b});
    }
};
}  // namespace

namespace {

void free_resampled(bp_handle* h) {
    cudaFree(h->lr_w); cudaFree(h->rf_w); cudaFree(h->mcm_w); cudaFree(h->rs_idx);
    h->lr_w = h->rf_w = h->mcm_w = nullptr;
    h->rs_idx = nullptr;
    h->Rw = 0;
    h->rs_num_host.clear();
    h->rs_den_host.clear();
}

void free_pool(bp_handle* h) {
    cudaFree(h->pool_prices); cudaFree(h->pool_caps); cudaFree(h->pool_hf); cudaFree(h->pool_rf);
    h->pool_prices = h->pool_caps = h->pool_hf = h->pool_rf = nullptr;
    h->pool_N = h->pool_D = 0;
    h->pool_R = 0;
}

void free_market(bp_handle* h) {
    free_resampled(h);
    cudaFree(h->prices); cudaFree(h->lr_d); cudaFree(h->caps); cudaFree(h->hf_prices);
    cudaFree(h->lr_hf); cudaFree(h->mcm); cudaFree(h->rf_row);
    h->prices = h->lr_d = h->caps = h->hf_prices = h->lr_hf = h->mcm = h->rf_row = nullptr;
    h->cap_daily = h->cap_hf = h->cap_mcm = h->cap_days = 0;
    h->has_market = false;
}

// Intraday return rows [row_begin, row_end) and their keep flags: every intraday log return goes through here, so that
// lr_hf and hf_keep always describe the same rows.  Price rows arrive in row order, so row row_begin - 1, which the first
// return row reads, is already resident.
int hf_returns(bp_handle* h, long long row_begin, long long row_end) {
    launch_hf_log_returns(h->hf_prices, h->N, h->lr_hf, h->ld, h->hf_keep.p, row_begin, row_end, h->N, h->sm_count, h->stream);
    h->launches++;
    CU_TRY(cudaGetLastError());
    return BP_OK;
}

// Conjugate stages read lr_hf.  The intraday prices arrive on the copy stream; their log returns are computed
// on the COMPUTE stream once the copy event has fired (a kernel on the copy stream would have to wait for
// free SMs behind the persistent Gram / solve kernels, and the next segment's copy would queue behind it).
int wait_hf(bp_handle* h) {
    if (h->hf_pending) {
        CU_TRY(cudaStreamWaitEvent(h->stream, h->ev_hf, 0));
        if (int rc = hf_returns(h, h->lr_hf_done, h->R)) return rc;
        h->lr_hf_done = h->R;
        h->hf_pending = false;
        h->seg_waited = h->n_seg;
    }
    return BP_OK;
}

// The same for a batch that reads intraday PRICE rows < rows_needed only: waits for the upload segments that cover them
// and computes their log returns; the later segments stay pending.  A caller that cuts a date-sorted batch into
// sub-batches along the segment boundaries thereby overlaps the compute of sub-batch k with the copy of segment k+1 on
// ANY path (the pipelined branch of run_batches does this inside one call, but only for the one-tile-per-day form).
int wait_hf_rows(bp_handle* h, long long rows_needed) {
    if (!h->hf_pending) return BP_OK;
    if (h->n_seg <= 1 || rows_needed >= h->R) return wait_hf(h);
    while (h->seg_waited < h->n_seg && h->lr_hf_done < rows_needed) {
        const int s = h->seg_waited;
        CU_TRY(cudaStreamWaitEvent(h->stream, h->ev_seg[s], 0));
        if (int rc = hf_returns(h, h->lr_hf_done, h->seg_end[s])) return rc;
        h->lr_hf_done = h->seg_end[s];
        h->seg_waited = s + 1;
    }
    if (h->seg_waited >= h->n_seg) {
        h->hf_pending = false;
        h->lr_hf_done = h->R;
    }
    return BP_OK;
}

int make_map(bp_handle* h, CUtensorMap* map, const double* base, long long rows, int ld) {
    // 3-D view (16-column group element, row, column group) of a row-major [rows][ld] matrix
    cuuint64_t dims[3] = {16, (cuuint64_t)rows, (cuuint64_t)(ld / 16)};
    cuuint64_t strides[2] = {(cuuint64_t)ld * sizeof(double), 16 * sizeof(double)};
    cuuint32_t box[3] = {16, (cuuint32_t)GRAM_KT, 8};
    cuuint32_t estr[3] = {1, 1, 1};
    CUresult r = h->encode(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT64, 3, const_cast<double*>(base), dims, strides, box,
                           estr, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B,
                           CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) return fail(BP_ERR_CUDA, "cuTensorMapEncodeTiled failed with CUresult %d", (int)r);
    return BP_OK;
}

// 2-D tensor map over a solver workspace of `rows` x ldS doubles (32-row x 16-column boxes)
int make_solve_map(bp_handle* h, CUtensorMap* map, const double* base, long long rows, int ldS) {
    cuuint64_t dims[2] = {(cuuint64_t)ldS, (cuuint64_t)rows};
    cuuint64_t strides[1] = {(cuuint64_t)ldS * sizeof(double)};
    cuuint32_t box[2] = {16, 32};
    cuuint32_t estr[2] = {1, 1};
    CUresult r = h->encode(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT64, 2, const_cast<double*>(base), dims, strides, box,
                           estr, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B,
                           CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) return fail(BP_ERR_CUDA, "cuTensorMapEncodeTiled (solver workspace) failed with CUresult %d", (int)r);
    return BP_OK;
}

// Grows buf to at least n elements, without keeping its contents; waits for the stream first, which may still read the
// old buffer.
template <class T>
int grow(bp_handle* h, DevBuf<T>& buf, size_t n) {
    if (n <= buf.cap) return BP_OK;
    if (buf.p) CU_TRY(cudaStreamSynchronize(h->stream));
    free_buf(buf);
    if (buf.pinned) CU_TRY(cudaHostAlloc(&buf.p, sizeof(T) * n, cudaHostAllocDefault));
    else CU_TRY(cudaMalloc(&buf.p, sizeof(T) * n));
    buf.cap = n;
    return BP_OK;
}

struct Chunk {
    // carved from the workspace for Wc windows
    double *S, *t, *pvec, *gvec, *rhs, *w0, *s0w0, *w1, *nu, *weights, *scal, *y, *mv;
    int* status;
};

Chunk carve(unsigned char* ws, const Layout& L, int Wc) {
    Chunk c;
    double* p = reinterpret_cast<double*>(ws);
    c.S = p;        p += (size_t)Wc * L.win_stride;
    c.t = p;        p += (size_t)Wc * L.ldv;
    c.pvec = p;     p += (size_t)Wc * L.ldv;
    c.gvec = p;     p += (size_t)Wc * L.ldv;
    c.rhs = p;      p += (size_t)Wc * L.ldv;
    c.w0 = p;       p += (size_t)Wc * L.ldv;
    c.s0w0 = p;     p += (size_t)Wc * L.ldv;
    c.w1 = p;       p += (size_t)Wc * L.ldv;
    c.nu = p;       p += (size_t)Wc * L.ldv;
    c.weights = p;  p += (size_t)Wc * L.ldv;
    c.scal = p;     p += (size_t)Wc * BP_NSCAL;
    c.y = p;        p += (size_t)Wc * L.y_stride;
    c.mv = p;       p += (size_t)Wc * L.mv_stride;
    c.status = reinterpret_cast<int*>(p);
    return c;
}

// the carved arrays as seen from window k of the chunk
Chunk chunk_at(const Chunk& c, const Layout& L, int k) {
    Chunk o = c;
    o.S += (size_t)k * L.win_stride;
    o.t += (size_t)k * L.ldv;       o.pvec += (size_t)k * L.ldv;  o.gvec += (size_t)k * L.ldv;
    o.rhs += (size_t)k * L.ldv;     o.w0 += (size_t)k * L.ldv;    o.s0w0 += (size_t)k * L.ldv;
    o.w1 += (size_t)k * L.ldv;      o.nu += (size_t)k * L.ldv;    o.weights += (size_t)k * L.ldv;
    o.scal += (size_t)k * BP_NSCAL;
    o.y += (size_t)k * L.y_stride;
    o.mv += (size_t)k * L.mv_stride;
    o.status += k;
    return o;
}

// validated, planned batch and its descriptor image on the device
struct Batch {
    BatchPlan plan;
    const int *day_row = nullptr, *span = nullptr, *hf_row0 = nullptr, *hf_span = nullptr;
    const int *extra_row = nullptr, *caps_row = nullptr;
    const int* gdesc = nullptr;        // [W][GRAM_DESC_INTS] Gram job descriptors
    const int* bdesc[2][2] = {{nullptr, nullptr}, {nullptr, nullptr}};   // block precompute launches [phase][level]
    const int* rdesc[2] = {nullptr, nullptr};      // phase B: [lo, hi) block ranges to pre-sum, per level
    const int* fdesc = nullptr;                    // phase B: [coarse, fineA, fineB] run ids to combine
    const int* hf_starts = nullptr;    // inner day blocks: price row where block k starts (nb + 1 entries)
    const int* hf_vids = nullptr;      // [W][3] scanned-vector ids of each window
    const double* prior_n = nullptr;
};

PlanCtx plan_ctx(const bp_handle* h) {
    PlanCtx c;
    c.has_market = h->has_market;
    c.N = h->N; c.ld = h->ld; c.D = h->D; c.Rw = h->Rw; c.n_mcm = h->n_mcm;
    c.R = h->R;
    c.hf_extra_rows = h->hf_extra_rows;
    c.has_caps = h->has_caps;
    c.has_mcm_w = h->mcm_w != nullptr;
    c.ws_limit = h->ws_limit;
    c.reuse_min_windows = h->reuse_min_windows;
    c.presum_min_days = h->presum_min_days;
    c.stacked = h->stacked;
    if (h->stacked) {
        c.n_blocks = (int)h->stack_day_start.size();
        c.day_block = h->stack_day_start.data();
        c.hf_block = h->stack_hf_start.empty() ? nullptr : h->stack_hf_start.data();
        c.rs_num = h->rs_num_host.empty() ? nullptr : h->rs_num_host.data();
        c.rs_den = h->rs_den_host.empty() ? nullptr : h->rs_den_host.data();
    }
    c.cond_estimate = h->cond_estimate;
    c.chain_group = h->chain_group;
    c.chain_max = chain_max_group();
    c.chain_smem_fits = chain_smem_bytes(h->N) <= (size_t)227 * 1024;
    c.hf_pending = h->hf_pending;
    c.n_seg = h->n_seg;
    c.seg_waited = h->seg_waited;
    return c;
}

// The descriptor image of the batch planned in out->plan, on the device
int upload_batch(bp_handle* h, const bp_window_batch* b, Batch* out) {
    const BatchPlan& P = out->plan;
    const int W = P.W;
    int rc;
    for (int ph = 0; ph < 2; ++ph)
        for (int l = 0; l < 2; ++l)
            if ((rc = grow(h, h->store[ph][l], P.store[ph][l]))) return rc;
    for (int l = 0; l < 2; ++l)
        if ((rc = grow(h, h->rstore[l], P.rstore[l]))) return rc;
    if ((rc = grow(h, h->fstore, P.fstore)) || (rc = grow(h, h->vstore, P.vstore))) return rc;
    const int slot = h->desc_turn ^= 1;
    if (h->ev_desc_armed[slot]) {
        CU_TRY(cudaEventSynchronize(h->ev_desc[slot]));      // its staging buffer has been fetched
        h->ev_desc_armed[slot] = false;
    }
    if ((rc = grow(h, h->desc_slot[slot], P.ints)) || (rc = grow(h, h->desc_host_slot[slot], P.ints))) return rc;
    int* dev = h->desc_slot[slot].p;
    write_batch(P, b, h->desc_host_slot[slot].p);
    // zero-copy fetch by a kernel on the compute stream (not the copy engine, see fetch_ints_kernel); the
    // staging buffer of this slot is rewritten two batches later, after this event
    launch_fetch_ints(h->desc_host_slot[slot].p, dev, (long long)P.ints, h->stream);
    h->launches++;
    CU_TRY(cudaGetLastError());
    if (!h->ev_desc[slot]) CU_TRY(cudaEventCreateWithFlags(&h->ev_desc[slot], cudaEventDisableTiming));
    CU_TRY(cudaEventRecord(h->ev_desc[slot], h->stream));
    h->ev_desc_armed[slot] = true;
    if (P.need_hf && b->prior_n) {
        if ((rc = grow(h, h->prior_n, (size_t)W))) return rc;
        CU_TRY(cudaMemcpyAsync(h->prior_n.p, b->prior_n, sizeof(double) * (size_t)W, cudaMemcpyHostToDevice, h->stream));
        CU_TRY(cudaStreamSynchronize(h->stream));
        out->prior_n = h->prior_n.p;
    }
    out->day_row = dev;
    out->span = dev + W;
    out->hf_row0 = dev + 3 * (size_t)W;
    out->hf_span = dev + 4 * (size_t)W;
    out->extra_row = P.resampled ? dev + 5 * (size_t)W : nullptr;
    out->caps_row = dev + 6 * (size_t)W;
    out->gdesc = dev + P.off_gram;
    for (int ph = 0; ph < 2; ++ph)
        for (int l = 0; l < 2; ++l) out->bdesc[ph][l] = P.phase[ph].nb[l] ? dev + P.off_blocks[ph][l] : nullptr;
    for (int l = 0; l < 2; ++l) out->rdesc[l] = P.nranges[l] ? dev + P.off_ranges[l] : nullptr;
    out->fdesc = P.nfull ? dev + P.off_triples : nullptr;
    out->hf_starts = P.phase[0].inner ? dev + P.off_starts : nullptr;
    out->hf_vids = P.presum ? dev + P.off_vids : nullptr;
    h->work_k_rows += P.work_k_rows;
    h->work_add_blocks += P.work_add_blocks;
    h->work_pre_rows += P.work_pre_rows;
    h->work_full_rows += P.work_full_rows;
    return BP_OK;
}

// The page-locked staging buffer of host-bound outputs, grown to `bytes`.  There is one: the previous copy out of it
// is drained first.
int host_stage(bp_handle* h, size_t bytes, double** p) {
    if (h->need_sync) {
        CU_TRY(cudaStreamSynchronize(h->stream));
        h->need_sync = false;
    }
    int rc = grow(h, h->stage, bytes);
    if (rc) return rc;
    *p = reinterpret_cast<double*>(h->stage.p);
    return BP_OK;
}

// dense copy of Wc windows' strided vectors ([Wc][N]) or symmetric matrices (sym: [Wc][N][N]) to dst, on the device
void unpack(bp_handle* h, const double* src, const Layout& L, int Wc, bool sym, double* dst) {
    if (sym) launch_unpack_sym(src, L.win_stride, L.ldS, L.N, Wc, dst, h->stream);
    else launch_unpack_vec(src, L.ldv, L.N, Wc, dst, h->stream);
    h->launches++;
}

// the same to a host or device destination; a host destination is reached through the staging buffer
int emit_dense(bp_handle* h, const double* src, const Layout& L, int Wc, bool sym, double* dst) {
    if (!dst) return BP_OK;
    if (is_device_ptr(dst)) {
        unpack(h, src, L, Wc, sym, dst);
        return BP_OK;
    }
    const size_t bytes = sizeof(double) * (size_t)Wc * L.N * (sym ? L.N : 1);
    double* stage = nullptr;
    int rc = host_stage(h, bytes, &stage);
    if (rc) return rc;
    unpack(h, src, L, Wc, sym, stage);
    CU_TRY(cudaMemcpyAsync(dst, stage, bytes, cudaMemcpyDeviceToHost, h->stream));
    h->need_sync = true;
    return BP_OK;
}

int emit_raw(bp_handle* h, const void* src, size_t bytes, void* dst) {
    if (!dst) return BP_OK;
    const bool dev = is_device_ptr(dst);
    CU_TRY(cudaMemcpyAsync(dst, src, bytes, dev ? cudaMemcpyDeviceToDevice : cudaMemcpyDeviceToHost, h->stream));
    if (!dev) h->need_sync = true;
    return BP_OK;
}

PrepParams prep_params(const bp_handle* h, const bp_window_batch* b, const Batch& B, const Layout& L, const Chunk& c,
                       int w0, int mode) {
    PrepParams p{};
    p.mode = mode;
    p.n_assets = h->N;
    p.n_window = B.plan.n;
    p.ld = h->ld;
    p.ldv = L.ldv;
    p.prior_kind = b->prior_weights == 0 ? BP_PRIOR_VW : BP_PRIOR_EW;
    p.mcm_scaling = b->mcm_scaling;
    p.lr_daily = B.plan.resampled ? h->lr_w : h->lr_d;
    p.lr_hf = h->lr_hf;
    p.hf_keep = h->hf_keep.p;
    p.caps = h->has_caps ? h->caps : nullptr;
    p.ld_caps = h->N;
    p.mcm = (mode == BP_MODE_CONJUGATE && h->mcm) ? h->mcm + (size_t)b->mcm_index * h->D : nullptr;
    if (B.plan.resampled) p.mcm = (mode == BP_MODE_CONJUGATE && h->mcm_w) ? h->mcm_w + (size_t)b->mcm_index * h->Rw : nullptr;
    p.mcm_rows = B.plan.mcm_rows;
    p.prior_n = B.prior_n ? B.prior_n + w0 : nullptr;
    p.rf_row = B.plan.resampled ? h->rf_w : h->rf_row;
    p.day_row = B.day_row + w0;
    p.extra_row = B.extra_row ? B.extra_row + w0 : nullptr;
    p.caps_row = B.caps_row ? B.caps_row + w0 : nullptr;
    p.span_days = B.span + w0;
    p.hf_row0 = B.hf_row0 + w0;
    p.hf_span = B.hf_span + w0;
    p.t = c.t; p.pvec = c.pvec; p.gvec = c.gvec; p.rhs = c.rhs; p.w0 = c.w0; p.s0w0 = c.s0w0;
    p.scal = c.scal;
    p.y_ws = c.y;
    p.y_stride = L.y_stride;
    p.hf_presum = (mode == BP_MODE_CONJUGATE && B.plan.presum) ? 1 : 0;
    p.hf_vsum = h->vstore.p;
    p.hf_vids = B.hf_vids ? B.hf_vids + 3 * (size_t)w0 : nullptr;
    p.use_band = B.plan.band_ok ? 1 : 0;
    p.band_ld = round_up(B.plan.n - 1, 2);
    p.band_aw = B.plan.band_ok ? h->band_aw.p + (size_t)w0 * p.band_ld : nullptr;
    p.band_stats = B.plan.band_ok ? h->band_stats.p + 2 * (size_t)w0 : nullptr;
    return p;
}

enum GramKind { GRAM_T, GRAM_S0, GRAM_S1, GRAM_J };

GramParams gram_params(const bp_handle* h, const Batch& B, const Layout& L, const Chunk& c, int w0, int Wc, GramKind kind) {
    GramParams g{};
    g.n_windows = Wc;
    g.n_assets = h->N;
    g.ldS = L.ldS;
    g.win_stride = L.win_stride;
    g.ldv = L.ldv;
    g.mirror = 0;
    g.scal = c.scal;
    g.out = c.S;
    g.desc = B.gdesc + (size_t)w0 * GRAM_DESC_INTS;
    for (int l = 0; l < 2; ++l) {
        g.store[0][l] = h->store[0][l].p;        // intraday: one tile per whole block
        g.store[1][l] = l == 0 ? h->fstore.p : h->rstore[l].p;      // daily: ONE combined tile per window (runs of whole blocks, pre-summed)
    }
    const bool hf = kind == GRAM_S0 || kind == GRAM_S1;
    const bool daily = kind != GRAM_S0;
    if (B.plan.presum) {
        g.store[0][1] = h->store[0][0].p;          // explicit tile ids into the unified [inner | suffix' | prefix] store
        if (hf) {
            g.mv_part = c.mv;
            g.mv_w0 = c.w0;
        }
    }
    g.use_phaseA = hf;
    g.use_phaseB = daily;
    if (hf) {
        g.use_alpha = 1;
        g.use_beta = 1;          // beta = alpha*m, g = hbar
        g.gvec = c.gvec;
    }
    if (daily) g.pvec = c.pvec;
    if (kind == GRAM_J) {
        g.use_beta = 1;          // beta = 1/n, g = t
        g.gvec = c.gvec;
    }
    return g;
}

// block precompute: the Gram tile of the whole blocks [k0[l], k1[l]) of a phase / level (default: all of them),
// written fragment-major into its store
int run_block_precompute(bp_handle* h, const Batch& B, int ph, const int* k0 = nullptr, const int* k1 = nullptr) {
    const int nt = (h->N + GRAM_TILE - 1) / GRAM_TILE;
    const size_t tile_doubles = (size_t)(nt * (nt + 1) / 2) * GRAM_BLOCK_TILE_DOUBLES;
    for (int l = 0; l < 2; ++l) {
        const int b0 = k0 ? k0[l] : 0, b1 = k1 ? k1[l] : B.plan.phase[ph].nb[l];
        if (b1 <= b0) continue;
        GramParams g{};
        g.n_windows = b1 - b0;
        g.n_assets = h->N;
        g.desc = B.bdesc[ph][l] + (size_t)b0 * GRAM_DESC_INTS;
        g.use_phaseA = ph == 0;
        g.use_phaseB = ph == 1;
        g.tile_store_out = 1;
        g.out = h->store[ph][l].p + (size_t)b0 * tile_doubles;
        StageTimer tm(h, BP_STAGE_GRAM);
        CU_TRY(launch_gram(g, h->map_hf, h->map_d, h->sm_count, h->stream));
        h->launches++;
        if (ph == 1 && B.plan.nranges[l] > 0) {
            launch_range_sum(h->store[1][l].p, B.rdesc[l], B.plan.nranges[l], nt * (nt + 1) / 2, h->rstore[l].p, h->stream);
            h->launches++;
            CU_TRY(cudaGetLastError());
        }
    }
    if (ph == 1 && !k0 && B.plan.nfull > 0) {
        StageTimer tm(h, BP_STAGE_GRAM);
        launch_combine_runs(h->rstore[0].p, h->rstore[1].p, B.fdesc, B.plan.nfull, nt * (nt + 1) / 2, h->fstore.p, h->stream);
        h->launches++;
        CU_TRY(cudaGetLastError());
    }
    return BP_OK;
}

int run_gram(bp_handle* h, const GramParams& g, bool resampled) {
    StageTimer tm(h, BP_STAGE_GRAM);
    CU_TRY(launch_gram(g, h->map_hf, resampled ? h->map_w : h->map_d, h->sm_count, h->stream));
    h->launches++;
    return BP_OK;
}

int finish(bp_handle* h) {
    if (h->need_sync && !h->async_outputs) {
        CU_TRY(cudaStreamSynchronize(h->stream));
        h->need_sync = false;
    }
    return BP_OK;
}

// The solver's size limit, checked before anything is uploaded or launched
int check_solver_size(int N, int estimator) {
    const int nrhs = estimator == BP_EST_JORION ? 2 : 1;
    const int max_n = chol_max_assets(nrhs);
    if (N > max_n)
        return fail(BP_ERR_INVALID, "the Cholesky solver supports at most %d assets with %d right-hand side%s; got %d", max_n,
                    nrhs, nrhs > 1 ? "s" : "", N);
    return BP_OK;
}

// Cholesky + solves of wn windows of the workspace, starting at c: CTA job q factorises window q * stride.  Shared by
// run_batches, bp_dense_posterior and bp_solve_batched.  c.scal must hold n1 for conjugate windows.
int solve_windows(bp_handle* h, const Chunk& c, const Layout& L, int wn, int stride, int mode, int estimator, int n_returns,
                  double inv_gamma) {
    if (wn <= 0) return BP_OK;
    SolveParams sp{};
    sp.n_windows = wn;
    sp.w_stride = stride;
    sp.n_assets = L.N;
    sp.ldS = L.ldS;
    sp.win_stride = L.win_stride;
    sp.ldv = L.ldv;
    sp.mode = mode;
    sp.estimator = estimator;
    sp.n_returns = n_returns;
    sp.inv_gamma = inv_gamma;
    sp.S = c.S;
    sp.rhs = c.rhs;
    sp.scal = c.scal;
    sp.w1 = c.w1;
    sp.nu = c.nu;
    sp.weights = c.weights;
    sp.status = c.status;
    CUtensorMap smap;
    int rc = make_solve_map(h, &smap, c.S, ((long long)(wn - 1) * stride + 1) * L.rowsS, L.ldS);
    if (rc) return rc;
    if (h->cond_estimate) {
        // anorm1 of the matrix the factorisation is about to overwrite
        StageTimer tm(h, BP_STAGE_COND);
        CU_TRY(launch_sym_norm1(sp, h->stream));
        h->launches++;
    }
    {
        StageTimer tm(h, BP_STAGE_SOLVE);
        CU_TRY(launch_chol_solve(sp, smap, h->sm_count, h->stream));
    }
    h->launches++;
    if (h->cond_estimate) {
        StageTimer tm(h, BP_STAGE_COND);
        CU_TRY(launch_chol_rcond(sp, h->stream));
        h->launches++;
    }
    h->work_factored += wn;
    return BP_OK;
}

// Cholesky + solves of wn windows of a batched call, from window k of the chunk at c; the reference evaluates
// (1/gamma) * nu (:836,:849)
int solve_batch_windows(bp_handle* h, const bp_window_batch* b, const Layout& L, const Chunk& c, const CallDesc& call, int k,
                        int wn, int stride = 1) {
    return solve_windows(h, chunk_at(c, L, k), L, wn, stride, call.mode, call.estimator, b->rolling_window - 1,
                         1.0 / b->risk_aversion);
}

// Outputs of the chunk's windows [w0, w0 + wc) of a batch of W windows, in one order: the solution when solved
// (weights, nu, w1, status), then t, w0 (with_w0), rhs and the scalars.  Shared by run_batches and bp_solve_batched.
int emit_chunk(bp_handle* h, const Chunk& c, const Layout& L, const bp_outputs* out, int w0, int wc, int W, bool solved,
               bool with_w0) {
    const size_t ov = (size_t)w0 * L.N;
    auto at = [ov](double* p) { return p ? p + ov : nullptr; };
    int rc;
    if (solved) {
        if ((rc = emit_dense(h, c.weights, L, wc, false, at(out->weights)))) return rc;
        if ((rc = emit_dense(h, c.nu, L, wc, false, at(out->nu)))) return rc;
        if ((rc = emit_dense(h, c.w1, L, wc, false, at(out->w1)))) return rc;
        if ((rc = emit_raw(h, c.status, sizeof(int) * (size_t)wc, out->status ? out->status + w0 : nullptr))) return rc;
    }
    if ((rc = emit_dense(h, c.t, L, wc, false, at(out->t)))) return rc;
    if (with_w0 && (rc = emit_dense(h, c.w0, L, wc, false, at(out->w0)))) return rc;
    if ((rc = emit_dense(h, c.rhs, L, wc, false, at(out->rhs)))) return rc;
    if ((rc = emit_raw(h, c.scal, sizeof(double) * (size_t)wc * BP_NSCAL,
                       out->scalars ? out->scalars + (size_t)w0 * BP_NSCAL : nullptr))) return rc;
    // the workspace is reused by the next chunk: host-bound copies must have drained
    if (w0 + wc < W && h->need_sync) {
        CU_TRY(cudaStreamSynchronize(h->stream));
        h->need_sync = false;
    }
    return BP_OK;
}

// Block precompute before the chunk loop: the gathered overnight returns and the intraday blocks (with their scans on
// the pre-summed path) of a conjugate batch, then the daily blocks
int run_blocks(bp_handle* h, const Batch& B, const CallDesc& call) {
    const BatchPlan& P = B.plan;
    const PhasePlan& A = P.phase[0];
    const bool conj = call.mode == BP_MODE_CONJUGATE;
    int rc;
    if (conj && A.inner && !P.presum) {
        launch_gather_rows_indexed(h->lr_hf, h->ld, B.hf_starts, h->R, 0, A.nb[0], h->stream);
        h->launches++;
        CU_TRY(cudaGetLastError());
    }
    if (conj && (call.S0 || call.S1 || call.solve || P.presum) && (rc = run_block_precompute(h, B, 0))) return rc;
    if (conj && P.presum) {
        // scans of the day blocks: column sums (vectors) and Gram tiles, suffix' and prefix per chunk
        StageTimer tm(h, BP_STAGE_GRAM);
        const int nt = (h->N + GRAM_TILE - 1) / GRAM_TILE;
        launch_block_col_sums(h->lr_hf, h->ld, B.hf_starts, 0, A.nb[0], h->vstore.p, h->stream);
        launch_vec_scan(h->vstore.p, h->ld, h->lr_hf, B.hf_starts, A.nb[0], A.chunk, h->stream);
        launch_tile_scan(h->store[0][0].p, nt * (nt + 1) / 2, nt, h->lr_hf, h->ld, B.hf_starts, A.nb[0], A.chunk, h->stream);
        h->launches += 3;
        CU_TRY(cudaGetLastError());
    }
    if ((call.T || call.S1 || call.solve) && (rc = run_block_precompute(h, B, 1))) return rc;
    return BP_OK;
}

// Window prep of the windows [w0, w0 + wc) of the batch; c: the workspace of window w0
int run_prep(bp_handle* h, const bp_window_batch* b, const Batch& B, const Layout& L, const Chunk& c, int w0, int wc,
             const CallDesc& call) {
    PrepParams pp = prep_params(h, b, B, L, c, w0, call.mode);
    if (call.estimator != BP_EST_NONE) pp.beta_den = B.plan.n - 1;       // sample covariance: centre with 1/m, m = n-1 returns
    {
        StageTimer tm(h, BP_STAGE_PREP);
        CU_TRY(launch_window_prep(pp, wc, h->stream, h->D));
        h->launches += pp.use_band ? (call.mode == BP_MODE_JEFFREYS ? 1 : 2) : 0;
    }
    h->launches++;
    return BP_OK;
}

// Pre-summed day blocks: S0 w0, v0, c and rhs are finished from the G w0 partials of the first Gram launch that
// contracts the intraday phase (it must precede the solve and every emit of rhs / scalars)
int run_post(bp_handle* h, const Layout& L, const Chunk& c, int wc) {
    PostParams q{};
    q.n_windows = wc;
    q.n_assets = L.N;
    q.ldv = L.ldv;
    q.mv_part = c.mv;
    q.w0 = c.w0;
    q.gvec = c.gvec;
    q.t = c.t;
    q.s0w0 = c.s0w0;
    q.rhs = c.rhs;
    q.scal = c.scal;
    StageTimer tm(h, BP_STAGE_PREP);
    CU_TRY(launch_conj_post(q, h->stream));
    h->launches++;
    return BP_OK;
}

// C = X_c'X_c  ->  m Sigma_LW / (1 - shrinkage) = C + rho I, rhs = t / (1 - shrinkage), in place (:727-729)
int run_shrink(bp_handle* h, const Batch& B, const Layout& L, const Chunk& c, int w0, int wc) {
    const BatchPlan& P = B.plan;
    ShrinkParams q{};
    q.n_windows = wc;
    q.n_assets = L.N;
    q.n_window = P.n;
    q.ld = h->ld;
    q.ldv = L.ldv;
    q.ldS = L.ldS;
    q.win_stride = L.win_stride;
    q.lr_daily = P.resampled ? h->lr_w : h->lr_d;
    q.rf_row = P.resampled ? h->rf_w : h->rf_row;
    q.day_row = B.day_row + w0;
    q.extra_row = B.extra_row ? B.extra_row + w0 : nullptr;
    q.span_days = B.span + w0;
    q.t = c.t;
    q.S = c.S;
    q.rhs = c.rhs;
    q.scal = c.scal;
    StageTimer tm(h, BP_STAGE_PREP);
    CU_TRY(launch_lw_shrink(q, h->stream));
    h->launches++;
    return BP_OK;
}

// S0 Gram of the chunk (intraday rows), finished by run_post when post; S0: its output or nullptr
int run_s0(bp_handle* h, const Batch& B, const Layout& L, const Chunk& c, int w0, int wc, bool post, double* S0) {
    int rc = run_gram(h, gram_params(h, B, L, c, w0, wc, GRAM_S0), B.plan.resampled);
    if (!rc && post) rc = run_post(h, L, c, wc);
    if (!rc) rc = emit_dense(h, c.S, L, wc, true, S0);
    return rc;
}

// S1 (conjugate) or J (Jeffreys) Gram of the chunk, of the base windows only on the chain path; finished by run_post
// when post, rewritten into the Ledoit-Wolf system for the shrinkage estimator; S1: its output or nullptr
int run_s1(bp_handle* h, const Batch& B, const Route& r, const Chunk& c, int w0, int wc, const CallDesc& call, bool post,
           double* S1) {
    GramParams gp = gram_params(h, B, r.L, c, w0, wc, call.mode == BP_MODE_CONJUGATE ? GRAM_S1 : GRAM_J);
    if (r.G >= 2) {                      // base windows only
        gp.w_stride = r.G;
        gp.n_windows = (wc + r.G - 1) / r.G;
    }
    int rc = run_gram(h, gp, B.plan.resampled);
    if (!rc && post) rc = run_post(h, r.L, c, wc);
    if (!rc && call.estimator == BP_EST_SHRINKAGE) rc = run_shrink(h, B, r.L, c, w0, wc);
    if (!rc) rc = emit_dense(h, c.S, r.L, wc, true, S1);
    return rc;
}

// Chain path: factorise the base windows of the chunk, then solve the other windows of each group relative to their base
int run_chain(bp_handle* h, const bp_window_batch* b, const Batch& B, const Route& r, const Chunk& c, int w0, int wc,
              const CallDesc& call) {
    const int G = r.G;
    int rc = solve_batch_windows(h, b, r.L, c, call, 0, (wc + G - 1) / G, G);
    if (rc) return rc;
    ChainParams cp{};
    cp.n_windows = wc;
    cp.group = G;
    cp.n_assets = h->N;
    cp.n_window = B.plan.n;
    cp.estimator = call.estimator;
    cp.ld = h->ld;
    cp.ldv = r.L.ldv;
    cp.ldS = r.L.ldS;
    cp.win_stride = r.L.win_stride;
    cp.inv_gamma = 1.0 / b->risk_aversion;
    cp.lr_daily = h->lr_d;
    cp.day_row = B.day_row + w0;
    cp.S = c.S;
    cp.t = c.t;
    cp.pvec = c.pvec;
    cp.w1 = c.w1;
    cp.nu = c.nu;
    cp.weights = c.weights;
    cp.scal = c.scal;
    cp.status = c.status;
    {
        StageTimer tm(h, BP_STAGE_CHAIN);
        CU_TRY(launch_jeffreys_chain(cp, h->stream));
    }
    h->launches++;
    h->work_chained += wc - (wc + G - 1) / G;
    return BP_OK;
}

// Pipelined conjugate batch (one workspace chunk) against a segmented asynchronous intraday upload: waits for the
// segments one by one, runs the prep + S1 Gram of the windows whose bars have arrived, and solves full waves of them
// between the segments.  *w_solved: the windows it solved.
int run_pipelined(bp_handle* h, const bp_window_batch* b, const Batch& B, const Route& r, const Chunk& c,
                  const CallDesc& call, double* S1, int* w_solved) {
    const BatchPlan& P = B.plan;
    const PhasePlan& A = P.phase[0];
    const Layout& L = r.L;
    const int N = h->N;
    int rc = run_block_precompute(h, B, 1);          // daily blocks do not wait for the bars
    if (rc) return rc;
    int w_done = 0, k_done[2] = {0, 0};
    *w_solved = 0;
    // S1 has to leave every segment's windows before the full waves below factorise them in place.  A device S1 is
    // unpacked straight into the output; a host S1 into the staging buffer (grown once, here), which is copied out
    // after the last segment, so that no segment waits for the host.
    double* s1_dev = nullptr;
    const size_t s1_bytes = sizeof(double) * (size_t)P.W * N * N;
    if (S1) {
        if (is_device_ptr(S1)) s1_dev = S1;
        else if ((rc = host_stage(h, s1_bytes, &s1_dev))) return rc;
    }
    for (int s = h->seg_waited; s < h->n_seg; ++s) {
        CU_TRY(cudaStreamWaitEvent(h->stream, h->ev_seg[s], 0));
        const bool last = s == h->n_seg - 1;
        const long long r_end = h->seg_end[s];
        if ((rc = hf_returns(h, h->lr_hf_done, r_end))) return rc;
        h->lr_hf_done = r_end;
        int k_ready[2];
        for (int l = 0; l < 2; ++l) {
            k_ready[l] = A.nb[l];
            if (!last && l == 0 && A.inner) {
                // day block k is complete once the bars below starts[k+1] have arrived
                const long long k = std::upper_bound(A.starts.begin() + 1, A.starts.end(), (int)std::min<long long>(r_end, 0x7fffffff)) -
                                    (A.starts.begin() + 1);
                k_ready[l] = (int)std::min<long long>(A.nb[l], std::max<long long>(k, k_done[l]));
            } else if (!last && A.blk[l] > 0) {
                const long long k = floor_div(r_end, A.blk[l]) - A.bmin[l];
                k_ready[l] = (int)std::min<long long>(A.nb[l], std::max<long long>(k, k_done[l]));
            }
        }
        if (A.inner) {
            launch_gather_rows_indexed(h->lr_hf, h->ld, B.hf_starts, h->R, k_done[0], k_ready[0], h->stream);
            h->launches++;
            CU_TRY(cudaGetLastError());
        }
        if ((rc = run_block_precompute(h, B, 0, k_done, k_ready))) return rc;
        k_done[0] = k_ready[0];
        k_done[1] = k_ready[1];
        int w_end = w_done;
        if (last) w_end = P.W;
        else while (w_end < P.W && (long long)b->hf_hi[w_end] <= r_end) ++w_end;
        if (w_end > w_done) {
            const Chunk cw = chunk_at(c, L, w_done);
            if ((rc = run_prep(h, b, B, L, cw, w_done, w_end - w_done, call))) return rc;
            if ((rc = run_gram(h, gram_params(h, B, L, cw, w_done, w_end - w_done, GRAM_S1), P.resampled))) return rc;
            if (s1_dev) {
                unpack(h, cw.S, L, w_end - w_done, true, s1_dev + (size_t)w_done * N * N);
                CU_TRY(cudaGetLastError());
            }
            w_done = w_end;
        }
        // Solve the full waves of windows that are ready: the compute stream would otherwise idle until the next
        // segment arrives (the copy takes longer than the statistics / Gram stages), and after the last segment
        // only the remainder (less than one wave) is left instead of every window.  Full waves cost nothing in
        // occupancy whichever of the copy and the GPU is the bottleneck.
        if (!last) {
            const int wave = chol_wave_windows(h->sm_count);
            // Full waves only -- a launch costs the latency of one factorisation however few windows it has -- except
            // before the LAST segment: whatever is ready then is solved while the last segment is on the bus, so that
            // only the last segment's own windows follow the copy (with the default plan that is a full wave anyway;
            // plans with several short tail segments were measured slower, windows.plan_wave_fractions)
            const bool before_last = s == h->n_seg - 2;
            const int wn = before_last ? w_done - *w_solved : (w_done - *w_solved) / wave * wave;
            if (wn > 0) {
                if ((rc = solve_batch_windows(h, b, L, c, call, *w_solved, wn))) return rc;
                *w_solved += wn;
            }
        }
    }
    if (s1_dev && s1_dev != S1) {
        CU_TRY(cudaMemcpyAsync(S1, s1_dev, s1_bytes, cudaMemcpyDeviceToHost, h->stream));
        h->need_sync = true;
    }
    h->seg_waited = h->n_seg;
    h->hf_pending = false;
    return BP_OK;
}

// Shared driver of bp_conjugate_batched / bp_jeffreys_batched / bp_estimator_batched / bp_stats_batched /
// bp_hf_cov_batched / bp_moments_batched: validate, plan, upload the descriptors, then run the stages
int run_batches(bp_handle* h, const bp_window_batch* b, const bp_outputs* out, int mode, bool solve, int estimator = BP_EST_NONE) {
    if (!h || !b) return fail(BP_ERR_INVALID, "null handle or batch");
    int rc;
    if (solve && h->has_market && (rc = check_solver_size(h->N, estimator))) return rc;
    const CallDesc call{mode, solve, estimator, out->T != nullptr, out->S0 != nullptr, out->S1 != nullptr};
    const bool conj = mode == BP_MODE_CONJUGATE;
    PlanCtx ctx = plan_ctx(h);
    if ((rc = check_batch(ctx, b, conj, &g_err)) || (rc = check_call(ctx, b, call, &g_err))) return rc;
    const int G = plan_chain_group(ctx, b, call);
    ctx.stride = G >= 2 ? G : 1;       // the chain path runs only the base windows through the Gram kernel
    Batch B;
    Route r;
    if ((rc = plan_batch(ctx, b, conj, &B.plan, &g_err)) || (rc = plan_route(ctx, B.plan, b, call, G, &r, &g_err))) return rc;
    const BatchPlan& P = B.plan;
    // every allocation / launch below must land on the handle's device, whatever the calling thread's current device
    // is (two handles on two GPUs in one thread, or torch having switched)
    CU_TRY(cudaSetDevice(h->device));
    if ((rc = upload_batch(h, b, &B))) return rc;
    if (r.hf_wait_rows > 0 && (rc = wait_hf_rows(h, r.hf_wait_rows))) return rc;
    if ((rc = grow(h, h->ws, (size_t)r.Wc * r.L.per_window + 256))) return rc;
    const Chunk c = carve(h->ws.p, r.L, r.Wc);
    if (P.band_ok && ((rc = grow(h, h->band_aw, (size_t)P.W * round_up(P.n - 1, 2))) ||
                      (rc = grow(h, h->band_stats, 2 * (size_t)P.W))))
        return rc;

    if ((call.T || call.S0 || call.S1 || solve) && !r.pipelined && (rc = run_blocks(h, B, call))) return rc;
    int w_solved = 0;          // windows already solved by the pipelined path (full waves, between the upload segments)
    if (r.pipelined && (rc = run_pipelined(h, b, B, r, c, call, out->S1, &w_solved))) return rc;
    const size_t NN = (size_t)h->N * h->N;
    const bool post = conj && P.presum;        // each chunk's first Gram launch of the intraday phase runs run_post
    for (int w0 = 0; w0 < P.W; w0 += r.Wc) {
        const int wc = std::min(r.Wc, P.W - w0);
        if (!r.pipelined && (rc = run_prep(h, b, B, r.L, c, w0, wc, call))) return rc;
        if (out->T && ((rc = run_gram(h, gram_params(h, B, r.L, c, w0, wc, GRAM_T), P.resampled)) ||
                       (rc = emit_dense(h, c.S, r.L, wc, true, out->T + w0 * NN))))
            return rc;
        const bool s0 = conj && (out->S0 || (post && !solve && !out->S1));
        if (s0 && (rc = run_s0(h, B, r.L, c, w0, wc, post, out->S0 ? out->S0 + w0 * NN : nullptr))) return rc;
        // (the pipelined path has run the S1 Gram and unpacked S1)
        if ((solve || out->S1) && !r.pipelined &&
            (rc = run_s1(h, B, r, c, w0, wc, call, post && !s0, out->S1 ? out->S1 + w0 * NN : nullptr)))
            return rc;
        if (solve && r.G >= 2 && (rc = run_chain(h, b, B, r, c, w0, wc, call))) return rc;
        if (solve && r.G < 2 && (rc = solve_batch_windows(h, b, r.L, c, call, w_solved, wc - w_solved))) return rc;
        if ((rc = emit_chunk(h, c, r.L, out, w0, wc, P.W, solve, conj))) return rc;
    }
    return finish(h);
}

}  // namespace

extern "C" {

const char* bp_last_error(void) { return g_err.c_str(); }
int bp_version(void) { return 100; }

int bp_init(int device, bp_handle** out) {
    if (!out) return fail(BP_ERR_INVALID, "out is null");
    *out = nullptr;
    int count = 0;
    if (cudaGetDeviceCount(&count) != cudaSuccess || count == 0) {
        cudaGetLastError();
        return fail(BP_ERR_NO_DEVICE, "no CUDA device visible: libbayes_portfolio has no CPU path");
    }
    if (device < 0 || device >= count) return fail(BP_ERR_INVALID, "device %d out of range (%d visible)", device, count);
    cudaDeviceProp prop;
    CU_TRY(cudaGetDeviceProperties(&prop, device));
    if (prop.major != 10)
        return fail(BP_ERR_NO_DEVICE, "device %d is sm_%d%d; this library is built for sm_100a only", device, prop.major, prop.minor);
    CU_TRY(cudaSetDevice(device));
    bp_handle* h = new bp_handle();
    h->device = device;
    h->sm_count = prop.multiProcessorCount;
    void* fn = nullptr;
    cudaDriverEntryPointQueryResult qres;
    cudaError_t e = cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qres);
    if (e != cudaSuccess || qres != cudaDriverEntryPointSuccess || !fn) {
        delete h;
        return fail(BP_ERR_CUDA, "cuTensorMapEncodeTiled entry point unavailable");
    }
    h->encode = reinterpret_cast<PFN_cuTensorMapEncodeTiled_v12000>(fn);
    if (cudaStreamCreateWithFlags(&h->copy_stream, cudaStreamNonBlocking) != cudaSuccess ||
        cudaEventCreateWithFlags(&h->ev_main, cudaEventDisableTiming) != cudaSuccess ||
        cudaEventCreateWithFlags(&h->ev_hf, cudaEventDisableTiming) != cudaSuccess) {
        delete h;
        return fail(BP_ERR_CUDA, "could not create the copy stream / events");
    }
    *out = h;
    return BP_OK;
}

int bp_destroy(bp_handle* h) {
    if (!h) return BP_OK;
    cudaSetDevice(h->device);
    cudaStreamSynchronize(h->stream);
    cudaStreamSynchronize(h->copy_stream);
    free_market(h);
    free_pool(h);
    free_buf(h->pool_cols);
    free_buf(h->hf_keep);
    cudaStreamDestroy(h->copy_stream);
    cudaEventDestroy(h->ev_main);
    cudaEventDestroy(h->ev_hf);
    for (cudaEvent_t e : h->ev_seg)
        if (e) cudaEventDestroy(e);
    for (int k = 0; k < 2; ++k) {
        free_buf(h->desc_slot[k]);
        free_buf(h->desc_host_slot[k]);
        if (h->ev_desc[k]) cudaEventDestroy(h->ev_desc[k]);
    }
    for (int a = 0; a < 2; ++a)
        for (int l = 0; l < 2; ++l) free_buf(h->store[a][l]);
    free_buf(h->rstore[0]);
    free_buf(h->rstore[1]);
    free_buf(h->fstore);
    free_buf(h->vstore);
    free_buf(h->prior_n);
    free_buf(h->band_aw);
    free_buf(h->stack_rows);
    free_buf(h->band_stats);
    free_buf(h->ws);
    free_buf(h->stage);
    for (cudaEvent_t e : h->ev_pool) cudaEventDestroy(e);
    if (h->ev_t0) cudaEventDestroy(h->ev_t0);
    delete h;
    return BP_OK;
}

int bp_set_stream(bp_handle* h, void* cuda_stream) {
    if (!h) return fail(BP_ERR_INVALID, "null handle");
    cudaStream_t st = reinterpret_cast<cudaStream_t>(cuda_stream);
    if (st != h->stream) {
        // work queued on the old stream still uses the shared workspace, staging buffer and descriptor slots
        CU_TRY(cudaSetDevice(h->device));
        CU_TRY(cudaStreamSynchronize(h->stream));
        h->need_sync = false;
        h->stream = st;
    }
    return BP_OK;
}

int bp_synchronize(bp_handle* h) {
    if (!h) return fail(BP_ERR_INVALID, "null handle");
    CU_TRY(cudaStreamSynchronize(h->copy_stream));
    CU_TRY(cudaStreamSynchronize(h->stream));
    h->need_sync = false;
    return BP_OK;
}

int bp_wait_upload(bp_handle* h) {
    if (!h) return fail(BP_ERR_INVALID, "null handle");
    CU_TRY(cudaSetDevice(h->device));
    if (h->has_market && h->R > 0) CU_TRY(cudaEventSynchronize(h->ev_hf));      // the intraday block (copy stream)
    return BP_OK;
}

int bp_set_async_outputs(bp_handle* h, int enable) {
    if (!h) return fail(BP_ERR_INVALID, "null handle");
    if (!enable && h->need_sync) {
        CU_TRY(cudaStreamSynchronize(h->stream));
        h->need_sync = false;
    }
    h->async_outputs = enable != 0;
    return BP_OK;
}

int bp_set_workspace_limit(bp_handle* h, size_t bytes) {
    if (!h) return fail(BP_ERR_INVALID, "null handle");
    h->ws_limit = bytes;
    return BP_OK;
}

int bp_device_info(bp_handle* h, int* sm_count, size_t* free_bytes, size_t* total_bytes) {
    if (!h) return fail(BP_ERR_INVALID, "null handle");
    CU_TRY(cudaSetDevice(h->device));
    size_t f = 0, t = 0;
    CU_TRY(cudaMemGetInfo(&f, &t));
    if (sm_count) *sm_count = h->sm_count;
    if (free_bytes) *free_bytes = f;
    if (total_bytes) *total_bytes = t;
    return BP_OK;
}

long long bp_launch_count(bp_handle* h) { return h ? h->launches : 0; }

int bp_get_gram_work(bp_handle* h, double* out4) {
    if (!h || !out4) return fail(BP_ERR_INVALID, "null argument");
    out4[0] = h->work_k_rows;       // window rows contracted on the tensor cores (padded to 8)
    out4[1] = h->work_add_blocks;   // precomputed block tiles added per tile pair
    out4[2] = h->work_pre_rows;     // rows contracted by the block precompute launches
    out4[3] = h->work_full_rows;    // rows a from-scratch contraction of every window would touch
    h->work_k_rows = h->work_add_blocks = h->work_pre_rows = h->work_full_rows = 0;
    return BP_OK;
}

int bp_set_jeffreys_chain(bp_handle* h, int group) {
    if (!h) return fail(BP_ERR_INVALID, "null handle");
    if (group < 0 || group > chain_max_group()) return fail(BP_ERR_INVALID, "group must be in [0, %d]", chain_max_group());
    h->chain_group = group;
    return BP_OK;
}

int bp_set_condition_estimate(bp_handle* h, int enable) {
    if (!h) return fail(BP_ERR_INVALID, "null handle");
    h->cond_estimate = enable != 0;
    return BP_OK;
}

int bp_get_solve_work(bp_handle* h, double* out2) {
    if (!h || !out2) return fail(BP_ERR_INVALID, "null argument");
    out2[0] = h->work_factored;
    out2[1] = h->work_chained;
    h->work_factored = h->work_chained = 0;
    return BP_OK;
}

int bp_set_hf_presum_min_days(bp_handle* h, int min_days) {
    if (!h) return fail(BP_ERR_INVALID, "null handle");
    if (min_days < 0) return fail(BP_ERR_INVALID, "min_days must be >= 0");
    h->presum_min_days = min_days;
    return BP_OK;
}

int bp_set_reuse_min_windows(bp_handle* h, int min_windows) {
    if (!h) return fail(BP_ERR_INVALID, "null handle");
    h->reuse_min_windows = min_windows;
    return BP_OK;
}

int bp_set_upload_pipeline(bp_handle* h, int segments, long long min_bytes) {
    if (!h) return fail(BP_ERR_INVALID, "null handle");
    if (segments < 1 || segments > bp_handle::MAX_SEG || min_bytes < 0)
        return fail(BP_ERR_INVALID, "segments must be in [1,%d] and min_bytes >= 0", bp_handle::MAX_SEG);
    h->pipe_segments = segments;
    h->pipe_min_bytes = (size_t)min_bytes;
    return BP_OK;
}

int bp_set_upload_fractions(bp_handle* h, int n, const double* cum_fractions) {
    if (!h) return fail(BP_ERR_INVALID, "null handle");
    if (n <= 0 || !cum_fractions) {
        h->n_frac = 0;
        return BP_OK;
    }
    if (n > bp_handle::MAX_SEG) return fail(BP_ERR_INVALID, "at most %d segments", bp_handle::MAX_SEG);
    double prev = 0.0;
    for (int i = 0; i < n; ++i) {
        if (!(cum_fractions[i] >= prev) || cum_fractions[i] > 1.0)
            return fail(BP_ERR_INVALID, "cumulative fractions must be non-decreasing in [0, 1]");
        prev = cum_fractions[i];
    }
    for (int i = 0; i < n; ++i) h->frac[i] = cum_fractions[i];
    h->n_frac = n;
    return BP_OK;
}

int bp_solve_wave_windows(bp_handle* h) {
    if (!h) return 0;
    if (cudaSetDevice(h->device) != cudaSuccess) return 0;      // the cluster occupancy query needs the handle's device
    return chol_wave_windows(h->sm_count);
}

int bp_set_stage_timing(bp_handle* h, int enable) {
    if (!h) return fail(BP_ERR_INVALID, "null handle");
    h->timing = enable != 0;
    return BP_OK;
}

int bp_get_stage_times(bp_handle* h, double* ms, long long* launches) {
    if (!h || !ms || !launches) return fail(BP_ERR_INVALID, "null argument");
    CU_TRY(cudaStreamSynchronize(h->stream));
    for (int i = 0; i < BP_NSTAGE; ++i) {
        ms[i] = 0.0;
        launches[i] = 0;
    }
    static const bool timeline = getenv("BP_TIMELINE") != nullptr;
    for (const auto& sp : h->spans) {
        float t = 0.f;
        CU_TRY(cudaEventElapsedTime(&t, sp.a, sp.b));
        ms[sp.stage] += (double)t;
        launches[sp.stage] += 1;
        if (timeline) {
            float t0 = 0.f;
            if (cudaEventElapsedTime(&t0, h->t0_armed ? h->ev_t0 : h->spans.front().a, sp.a) != cudaSuccess) t0 = -1.f;
            fprintf(stderr, "[timeline] stage %d start %8.3f ms dur %7.3f ms\n", sp.stage, t0, t);
        }
    }
    (void)cudaGetLastError();
    h->spans.clear();
    h->ev_used = 0;
    return BP_OK;
}

int bp_prepare_market(bp_handle* h) {
    if (!h) return fail(BP_ERR_INVALID, "null handle");
    if (!h->has_market) return fail(BP_ERR_STATE, "no market uploaded");
    CU_TRY(cudaSetDevice(h->device));
    int rc = wait_hf(h);
    if (rc) return rc;
    {
        StageTimer tm(h, BP_STAGE_LOGRET);
        launch_log_returns(h->prices, h->N, h->lr_d, h->ld, h->D, h->N, h->sm_count, h->stream);
        h->launches++;
        if (h->R > 0 && (rc = hf_returns(h, 0, h->R))) return rc;
    }
    CU_TRY(cudaGetLastError());
    return BP_OK;
}

// Shared body of bp_upload_market / bp_upload_market_async.  Device buffers are reused when the new
// market fits the allocated capacity; the host arrays are copied in their dense layout with plain 1-D
// copies (full PCIe rate from pinned memory) and padded on the fly by the log-return kernel.  The
// intraday block (by far the largest) goes over a second stream together with its log-return kernel,
// so stages that do not read it (Jeffreys, daily statistics) overlap the transfer.
// Working-market buffers for N columns, D daily rows, R intraday rows (grown when needed) and the bookkeeping every
// way of filling them shares (host upload, device gather from the pool)
static int begin_market(bp_handle* h, int N, int D, long long R, int n_mcm) {
    const int ld = round_up(N, 16);
    const size_t need_daily = (size_t)D * ld, need_hf = (size_t)R * ld, need_mcm = (size_t)std::max(n_mcm, 1) * D;
    if (need_daily > h->cap_daily || need_hf > h->cap_hf || need_mcm > h->cap_mcm || (size_t)D > h->cap_days) {
        // grow: everything in flight must be done with the old buffers
        CU_TRY(cudaStreamSynchronize(h->stream));
        CU_TRY(cudaStreamSynchronize(h->copy_stream));
        free_market(h);
        CU_TRY(cudaMalloc(&h->prices, sizeof(double) * need_daily));
        CU_TRY(cudaMalloc(&h->lr_d, sizeof(double) * need_daily));
        CU_TRY(cudaMalloc(&h->caps, sizeof(double) * need_daily));
        CU_TRY(cudaMalloc(&h->rf_row, sizeof(double) * (size_t)D));
        CU_TRY(cudaMalloc(&h->mcm, sizeof(double) * need_mcm));
        if (need_hf) {
            CU_TRY(cudaMalloc(&h->hf_prices, sizeof(double) * need_hf));
            h->lr_hf_ld_cap = ld;
            h->lr_hf_rows_cap = R + R / 8 + 64;        // + room for the gathered overnight rows
            CU_TRY(cudaMalloc(&h->lr_hf, sizeof(double) * (size_t)h->lr_hf_rows_cap * ld));
        }
        h->cap_daily = need_daily;
        h->cap_hf = need_hf;
        h->cap_mcm = need_mcm;
        h->cap_days = (size_t)D;
    }
    if (h->lr_w) {
        // resampled rows refer to the previous prices
        CU_TRY(cudaStreamSynchronize(h->stream));
        free_resampled(h);
    }
    if (int rc = grow(h, h->hf_keep, (size_t)R)) return rc;
    h->N = N; h->D = D; h->ld = ld; h->R = R; h->n_mcm = n_mcm;
    if (h->timing) {
        if (!h->ev_t0) CU_TRY(cudaEventCreate(&h->ev_t0));
        CU_TRY(cudaEventRecord(h->ev_t0, h->stream));
        h->t0_armed = true;
    }
    h->n_seg = 0;
    h->seg_waited = 0;
    h->lr_hf_done = 0;
    h->hf_pending = false;
    h->stacked = false;
    h->stack_day_start.clear();
    h->stack_hf_start.clear();
    return BP_OK;
}

// daily log returns and the tensor maps of the (filled or being filled) working market
static int finish_market(bp_handle* h) {
    const int N = h->N, D = h->D, ld = h->ld;
    const long long R = h->R;
    int rc;
    launch_log_returns(h->prices, N, h->lr_d, ld, D, N, h->sm_count, h->stream);
    h->launches++;
    CU_TRY(cudaGetLastError());
    if ((rc = make_map(h, &h->map_d, h->lr_d, D, ld))) return rc;
    if (R > 0) {
        // rows available behind the R return rows at the CURRENT leading dimension
        h->hf_extra_rows = (long long)((size_t)h->lr_hf_rows_cap * h->lr_hf_ld_cap / ld) - R;
        if (h->hf_extra_rows < 0) h->hf_extra_rows = 0;
        if ((rc = make_map(h, &h->map_hf, h->lr_hf, R + h->hf_extra_rows, ld))) return rc;
    } else {
        h->map_hf = h->map_d;
    }
    h->has_market = true;
    return BP_OK;
}

// the checks the working market (noun "market") and the pool (noun "pool") share; the pool ignores mcm
static int check_market_desc(const bp_market_desc* m, const char* noun) {
    if (m->n_assets <= 0 || m->n_days < 2 || !m->prices || !m->rf_row)
        return fail(BP_ERR_INVALID, "%s needs n_assets > 0, n_days >= 2, prices and rf_row", noun);
    if (m->n_hf_rows < 0 || (m->n_hf_rows > 0 && !m->hf_prices)) return fail(BP_ERR_INVALID, "hf_prices missing");
    if (m->n_hf_rows > 0x7fffffffLL) return fail(BP_ERR_INVALID, "too many intraday rows for int32 row indices");
    return BP_OK;
}

static int upload_market_impl(bp_handle* h, const bp_market_desc* m, bool blocking) {
    if (!h || !m) return fail(BP_ERR_INVALID, "null handle or market");
    if (int rc = check_market_desc(m, "market")) return rc;
    if (m->n_mcm < 0 || (m->n_mcm > 0 && !m->mcm)) return fail(BP_ERR_INVALID, "mcm missing");
    CU_TRY(cudaSetDevice(h->device));
    const int N = m->n_assets, D = m->n_days;
    const long long R = m->n_hf_rows;
    int rc;
    if ((rc = begin_market(h, N, D, R, m->n_mcm))) return rc;
    h->has_caps = m->caps != nullptr;
    cudaStream_t st = h->stream;
    // the copy stream must not overwrite buffers that earlier launches on the compute stream still read
    CU_TRY(cudaEventRecord(h->ev_main, st));
    CU_TRY(cudaStreamWaitEvent(h->copy_stream, h->ev_main, 0));
    // small daily arrays first: both streams share one host->device copy engine, which serves copies in
    // issue order, and the Jeffreys / daily stages must not queue behind the 1.6 GB intraday block
    CU_TRY(cudaMemcpyAsync(h->prices, m->prices, sizeof(double) * (size_t)D * N, cudaMemcpyHostToDevice, st));
    if (m->caps) CU_TRY(cudaMemcpyAsync(h->caps, m->caps, sizeof(double) * (size_t)D * N, cudaMemcpyHostToDevice, st));
    if (m->n_mcm > 0)
        CU_TRY(cudaMemcpyAsync(h->mcm, m->mcm, sizeof(double) * (size_t)m->n_mcm * D, cudaMemcpyHostToDevice, st));
    CU_TRY(cudaMemcpyAsync(h->rf_row, m->rf_row, sizeof(double) * (size_t)D, cudaMemcpyHostToDevice, st));
    if (R > 0) {
        // asynchronous uploads of a large block go in segments with an event each; the log returns of a segment
        // are computed on the compute stream by its first consumer (wait_hf / the pipelined conjugate path)
        int nseg = 1;
        if (!blocking && sizeof(double) * (size_t)R * N >= h->pipe_min_bytes && R >= 64)
            nseg = h->n_frac > 0 ? h->n_frac : h->pipe_segments;
        // geometric segments (1/2, 1/4, ... of the rows): whatever the compute stream is busy with when the copy
        // starts, little work is left to do after the LAST segment has arrived
        long long r1 = 0;
        for (int s = 0; s < nseg; ++s) {
            const long long r0 = r1;
            r1 = s == nseg - 1 ? R : std::max(r0, R - (R >> (s + 1)));
            if (h->n_frac > 0 && s < nseg - 1)
                r1 = std::min<long long>(R, std::max<long long>(r0, (long long)std::ceil(h->frac[s] * (double)R)));
            CU_TRY(cudaMemcpyAsync(h->hf_prices + (size_t)r0 * N, m->hf_prices + (size_t)r0 * N, sizeof(double) * (size_t)(r1 - r0) * N,
                                   cudaMemcpyHostToDevice, h->copy_stream));
            if (nseg > 1) {
                if (!h->ev_seg[s]) CU_TRY(cudaEventCreateWithFlags(&h->ev_seg[s], cudaEventDisableTiming));
                CU_TRY(cudaEventRecord(h->ev_seg[s], h->copy_stream));
                h->seg_end[s] = r1;
            }
        }
        h->n_seg = nseg > 1 ? nseg : 0;
        CU_TRY(cudaEventRecord(h->ev_hf, h->copy_stream));
        h->hf_pending = true;
    }
    if ((rc = finish_market(h))) return rc;
    if (blocking) {
        // the caller's host arrays may be pageable and may be freed after return
        CU_TRY(cudaStreamSynchronize(h->copy_stream));
        CU_TRY(cudaStreamSynchronize(st));
    }
    return BP_OK;
}

int bp_path_metrics(bp_handle* h, int n_paths, int n_obs, const double* returns, const double* excess, double years,
                    double* out) {
    if (!h || !returns || !excess || !out) return fail(BP_ERR_INVALID, "null handle or array");
    if (n_paths <= 0 || n_obs < 2) return fail(BP_ERR_INVALID, "need at least one series of two returns");
    if (!(years > 0.0)) return fail(BP_ERR_INVALID, "years must be positive");
    CU_TRY(cudaSetDevice(h->device));
    const size_t n = (size_t)n_paths * n_obs;
    int rc = grow(h, h->stage, sizeof(double) * (2 * n + (size_t)n_paths * BP_PM_COUNT));
    if (rc) return rc;
    double* d = reinterpret_cast<double*>(h->stage.p);
    cudaStream_t st = h->stream;
    CU_TRY(cudaMemcpyAsync(d, returns, sizeof(double) * n, cudaMemcpyHostToDevice, st));
    CU_TRY(cudaMemcpyAsync(d + n, excess, sizeof(double) * n, cudaMemcpyHostToDevice, st));
    PathMetricsParams p{};
    p.n_paths = n_paths; p.n_obs = n_obs; p.ld = n_obs;
    p.returns = d; p.excess = d + n; p.years = years; p.out = d + 2 * n;
    CU_TRY(launch_path_metrics(p, st));
    h->launches++;
    CU_TRY(cudaMemcpyAsync(out, d + 2 * n, sizeof(double) * (size_t)n_paths * BP_PM_COUNT, cudaMemcpyDeviceToHost, st));
    CU_TRY(cudaStreamSynchronize(st));
    return BP_OK;
}

int bp_upload_pool(bp_handle* h, const bp_market_desc* m) {
    if (!h) return fail(BP_ERR_INVALID, "null handle");
    CU_TRY(cudaSetDevice(h->device));
    CU_TRY(cudaStreamSynchronize(h->stream));            // earlier gathers may still read the old pool
    free_pool(h);
    if (!m) return BP_OK;                                  // a null market releases the pool
    if (int rc = check_market_desc(m, "pool")) return rc;
    const size_t N = (size_t)m->n_assets, D = (size_t)m->n_days, R = (size_t)m->n_hf_rows;
    cudaStream_t st = h->stream;
    CU_TRY(cudaMalloc(&h->pool_prices, sizeof(double) * D * N));
    CU_TRY(cudaMalloc(&h->pool_rf, sizeof(double) * D));
    CU_TRY(cudaMemcpyAsync(h->pool_prices, m->prices, sizeof(double) * D * N, cudaMemcpyHostToDevice, st));
    CU_TRY(cudaMemcpyAsync(h->pool_rf, m->rf_row, sizeof(double) * D, cudaMemcpyHostToDevice, st));
    if (m->caps) {
        CU_TRY(cudaMalloc(&h->pool_caps, sizeof(double) * D * N));
        CU_TRY(cudaMemcpyAsync(h->pool_caps, m->caps, sizeof(double) * D * N, cudaMemcpyHostToDevice, st));
    }
    if (R > 0) {
        CU_TRY(cudaMalloc(&h->pool_hf, sizeof(double) * R * N));
        CU_TRY(cudaMemcpyAsync(h->pool_hf, m->hf_prices, sizeof(double) * R * N, cudaMemcpyHostToDevice, st));
    }
    CU_TRY(cudaStreamSynchronize(st));                    // the host arrays may be pageable / freed after return
    h->pool_N = m->n_assets;
    h->pool_D = m->n_days;
    h->pool_R = m->n_hf_rows;
    return BP_OK;
}

// The device half of every pool selection: window w's daily pool rows [tab[3w], tab[3w] + tab[3w+2]) in its columns
// cols[w][0..N) go to working rows tab[3w+1] on, its intraday rows likewise by the [W][3] table behind (tab[3W..6W)).
// The caller has checked columns and rows, and that the blocks tile the working market in window order.
static int gather_pool(bp_handle* h, int W, int N, const int* cols, const std::vector<long long>& tab) {
    long long D = 0, R = 0, max_d = 0, max_r = 0;
    for (int w = 0; w < W; ++w) {
        const long long nd = tab[3 * (size_t)w + 2], nh = tab[3 * ((size_t)W + w) + 2];
        D += nd;
        R += nh;
        max_d = std::max(max_d, nd);
        max_r = std::max(max_r, nh);
    }
    CU_TRY(cudaSetDevice(h->device));
    int rc;
    if ((rc = begin_market(h, N, (int)D, R, 0))) return rc;
    h->has_caps = h->pool_caps != nullptr;
    cudaStream_t st = h->stream;
    if ((rc = grow(h, h->pool_cols, (size_t)W * N)) || (rc = grow(h, h->stack_rows, tab.size()))) return rc;
    // (pageable host memory: the copies are staged before the call returns, so the caller's arrays may go away; stream
    // order keeps earlier gathers, which read the previous lists, ahead of them)
    CU_TRY(cudaMemcpyAsync(h->pool_cols.p, cols, sizeof(int) * (size_t)W * N, cudaMemcpyHostToDevice, st));
    CU_TRY(cudaMemcpyAsync(h->stack_rows.p, tab.data(), sizeof(long long) * tab.size(), cudaMemcpyHostToDevice, st));
    const long long pN = h->pool_N;
    const long long* day_tab = h->stack_rows.p;
    launch_gather_window_blocks(h->pool_prices, pN, h->prices, N, W, h->pool_cols.p, day_tab, max_d, st);
    h->launches++;
    if (h->pool_caps) {
        launch_gather_window_blocks(h->pool_caps, pN, h->caps, N, W, h->pool_cols.p, day_tab, max_d, st);
        h->launches++;
    }
    launch_gather_window_blocks(h->pool_rf, 1, h->rf_row, 1, W, nullptr, day_tab, max_d, st);
    h->launches++;
    if (R > 0) {
        launch_gather_window_blocks(h->pool_hf, pN, h->hf_prices, N, W, h->pool_cols.p, day_tab + 3 * (size_t)W, max_r, st);
        h->launches++;
        CU_TRY(cudaEventRecord(h->ev_hf, st));
        h->hf_pending = true;            // the first consumer computes the intraday log returns (wait_hf)
    }
    CU_TRY(cudaGetLastError());
    return finish_market(h);
}

int bp_select_market(bp_handle* h, const bp_pool_select* s) {
    if (!h || !s) return fail(BP_ERR_INVALID, "null handle or selection");
    if (!h->pool_prices) return fail(BP_ERR_STATE, "no pool resident: call bp_upload_pool first");
    if (s->n_cols <= 0 || !s->cols) return fail(BP_ERR_INVALID, "selection needs at least one column");
    if (s->day_lo < 0 || s->day_hi > h->pool_D || s->day_hi - s->day_lo < 2)
        return fail(BP_ERR_INVALID, "daily row range [%d, %d) outside the pool's %d rows (or shorter than 2)", s->day_lo, s->day_hi, h->pool_D);
    if (s->hf_lo < 0 || s->hf_hi < s->hf_lo || s->hf_hi > h->pool_R)
        return fail(BP_ERR_INVALID, "intraday row range outside the pool");
    for (int j = 0; j < s->n_cols; ++j)
        if (s->cols[j] < 0 || s->cols[j] >= h->pool_N) return fail(BP_ERR_INVALID, "column %d outside the pool's %d columns", s->cols[j], h->pool_N);
    // one window: a stack of one block
    return gather_pool(h, 1, s->n_cols, s->cols, {s->day_lo, 0, s->day_hi - s->day_lo, s->hf_lo, 0, s->hf_hi - s->hf_lo});
}

int bp_select_windows(bp_handle* h, const bp_window_select* s) {
    if (!h || !s) return fail(BP_ERR_INVALID, "null handle or selection");
    if (!h->pool_prices) return fail(BP_ERR_STATE, "no pool resident: call bp_upload_pool first");
    const int W = s->n_windows, N = s->n_cols;
    if (W <= 0 || N <= 0 || !s->cols || !s->day_lo || !s->day_hi || !s->day_off)
        return fail(BP_ERR_INVALID, "selection needs windows, columns and daily row ranges with their offsets");
    const bool with_hf = s->hf_lo || s->hf_hi || s->hf_off;
    if (with_hf && (!s->hf_lo || !s->hf_hi || !s->hf_off))
        return fail(BP_ERR_INVALID, "intraday row ranges need hf_lo, hf_hi and hf_off");
    if (N > h->pool_N) return fail(BP_ERR_INVALID, "%d columns per window: the pool has %d", N, h->pool_N);
    // [W][3] daily blocks, then [W][3] intraday blocks: (first pool row, first stack row, rows)
    std::vector<long long> tab(6 * (size_t)W, 0);
    long long D = 0, R = 0;
    for (int w = 0; w < W; ++w) {
        const int* c = s->cols + (size_t)w * N;
        for (int j = 0; j < N; ++j)
            if (c[j] < 0 || c[j] >= h->pool_N)
                return fail(BP_ERR_INVALID, "window %d: column %d outside the pool's %d columns", w, c[j], h->pool_N);
        const int lo = s->day_lo[w], hi = s->day_hi[w];
        if (lo < 0 || hi > h->pool_D || hi <= lo)
            return fail(BP_ERR_INVALID, "window %d: daily row range [%d, %d) outside the pool's %d rows (or empty)", w, lo, hi, h->pool_D);
        if (s->day_off[w] != D)
            return fail(BP_ERR_INVALID, "window %d: daily block starts at stack row %d, the blocks before it end at %lld: the blocks must tile the stack",
                        w, s->day_off[w], D);
        tab[3 * (size_t)w] = lo;
        tab[3 * (size_t)w + 1] = D;
        tab[3 * (size_t)w + 2] = hi - lo;
        D += hi - lo;
        if (D > 0x7fffffffLL) return fail(BP_ERR_INVALID, "too many daily rows in the stack for int32 row indices");
        if (!with_hf) continue;
        const long long hlo = s->hf_lo[w], hhi = s->hf_hi[w];
        if (hlo < 0 || hhi < hlo || hhi > h->pool_R)
            return fail(BP_ERR_INVALID, "window %d: intraday row range [%lld, %lld) outside the pool's %lld rows", w, hlo, hhi, h->pool_R);
        if (s->hf_off[w] != R)
            return fail(BP_ERR_INVALID, "window %d: intraday block starts at stack row %lld, the blocks before it end at %lld: the blocks must tile the stack",
                        w, s->hf_off[w], R);
        tab[3 * ((size_t)W + w)] = hlo;
        tab[3 * ((size_t)W + w) + 1] = R;
        tab[3 * ((size_t)W + w) + 2] = hhi - hlo;
        R += hhi - hlo;
        if (R > 0x7fffffffLL) return fail(BP_ERR_INVALID, "too many intraday rows in the stack for int32 row indices");
    }
    if (D < 2) return fail(BP_ERR_INVALID, "the stack needs at least 2 daily rows");
    int rc;
    if ((rc = gather_pool(h, W, N, s->cols, tab))) return rc;
    h->stacked = true;
    h->stack_day_start.resize(W);
    h->stack_hf_start.resize(with_hf ? W : 0);
    for (int w = 0; w < W; ++w) {
        h->stack_day_start[w] = tab[3 * (size_t)w + 1];
        if (with_hf) h->stack_hf_start[w] = tab[3 * ((size_t)W + w) + 1];
    }
    return BP_OK;
}

int bp_upload_market(bp_handle* h, const bp_market_desc* m) { return upload_market_impl(h, m, true); }

int bp_upload_market_async(bp_handle* h, const bp_market_desc* m) { return upload_market_impl(h, m, false); }

int bp_set_resampled(bp_handle* h, const bp_resampled_desc* r) {
    if (!h || !r) return fail(BP_ERR_INVALID, "null argument");
    if (!h->has_market) return fail(BP_ERR_STATE, "no market uploaded");
    if (r->n_rows < 2 || !r->num_row || !r->den_row || !r->rf_row) return fail(BP_ERR_INVALID, "bp_resampled_desc incomplete");
    for (int i = 0; i < r->n_rows; ++i)
        if (r->num_row[i] < 0 || r->num_row[i] >= h->D || r->den_row[i] < 0 || r->den_row[i] >= h->D)
            return fail(BP_ERR_INVALID, "resampled row %d references a price row outside [0,%d)", i, h->D);
    CU_TRY(cudaSetDevice(h->device));
    CU_TRY(cudaStreamSynchronize(h->stream));
    free_resampled(h);
    const int Rw = r->n_rows;
    CU_TRY(cudaMalloc(&h->lr_w, sizeof(double) * (size_t)Rw * h->ld));
    CU_TRY(cudaMalloc(&h->rf_w, sizeof(double) * (size_t)Rw));
    CU_TRY(cudaMalloc(&h->rs_idx, sizeof(int) * 2 * (size_t)Rw));
    CU_TRY(cudaMemcpyAsync(h->rs_idx, r->num_row, sizeof(int) * (size_t)Rw, cudaMemcpyHostToDevice, h->stream));
    CU_TRY(cudaMemcpyAsync(h->rs_idx + Rw, r->den_row, sizeof(int) * (size_t)Rw, cudaMemcpyHostToDevice, h->stream));
    CU_TRY(cudaMemcpyAsync(h->rf_w, r->rf_row, sizeof(double) * (size_t)Rw, cudaMemcpyHostToDevice, h->stream));
    if (r->mcm && h->n_mcm > 0) {
        CU_TRY(cudaMalloc(&h->mcm_w, sizeof(double) * (size_t)h->n_mcm * Rw));
        CU_TRY(cudaMemcpyAsync(h->mcm_w, r->mcm, sizeof(double) * (size_t)h->n_mcm * Rw, cudaMemcpyHostToDevice, h->stream));
    }
    launch_gather_log_returns(h->prices, h->N, h->rs_idx, h->rs_idx + Rw, h->lr_w, h->ld, Rw, h->N, h->stream);
    h->launches++;
    CU_TRY(cudaGetLastError());
    h->Rw = Rw;
    if (h->stacked) {
        h->rs_num_host.assign(r->num_row, r->num_row + Rw);
        h->rs_den_host.assign(r->den_row, r->den_row + Rw);
    }
    int rc = make_map(h, &h->map_w, h->lr_w, Rw, h->ld);
    if (rc) return rc;
    CU_TRY(cudaStreamSynchronize(h->stream));     // host index arrays may be freed after return
    return BP_OK;
}

int bp_conjugate_batched(bp_handle* h, const bp_window_batch* b, const bp_outputs* out) {
    if (!out) return fail(BP_ERR_INVALID, "outputs missing");
    return run_batches(h, b, out, BP_MODE_CONJUGATE, true);
}

int bp_jeffreys_batched(bp_handle* h, const bp_window_batch* b, const bp_outputs* out) {
    if (!out) return fail(BP_ERR_INVALID, "outputs missing");
    return run_batches(h, b, out, BP_MODE_JEFFREYS, true);
}

int bp_estimator_batched(bp_handle* h, const bp_window_batch* b, int estimator, const bp_outputs* out) {
    if (!h || !b || !out) return fail(BP_ERR_INVALID, "null argument");
    if (estimator != BP_EST_JORION && estimator != BP_EST_SHRINKAGE)
        return fail(BP_ERR_INVALID, "estimator must be BP_ESTIMATOR_JORION or BP_ESTIMATOR_SHRINKAGE");
    if (out->T || out->S0) return fail(BP_ERR_INVALID, "estimator batches do not return T / S0 (use bp_stats_batched)");
    return run_batches(h, b, out, BP_MODE_JEFFREYS, true, estimator);
}

int bp_stats_batched(bp_handle* h, const bp_window_batch* b, double* t, double* T) {
    bp_outputs o;
    memset(&o, 0, sizeof(o));
    o.t = t;
    o.T = T;
    return run_batches(h, b, &o, BP_MODE_JEFFREYS, false);
}

int bp_hf_cov_batched(bp_handle* h, const bp_window_batch* b, double* n0, double* S0) {
    if (!h || !b) return fail(BP_ERR_INVALID, "null handle or batch");
    bp_outputs o;
    memset(&o, 0, sizeof(o));
    o.S0 = S0;
    std::vector<double> scal;
    if (n0) {
        scal.resize((size_t)std::max(b->n_windows, 0) * BP_NSCAL);
        o.scalars = scal.data();
    }
    int rc = run_batches(h, b, &o, BP_MODE_CONJUGATE, false);
    if (rc) return rc;
    if (n0) {
        if (is_device_ptr(n0)) return fail(BP_ERR_INVALID, "bp_hf_cov_batched: n0 must be a host pointer");
        for (int w = 0; w < b->n_windows; ++w) n0[w] = scal[(size_t)w * BP_NSCAL + BP_SCAL_N0];
    }
    return BP_OK;
}

int bp_moments_batched(bp_handle* h, const bp_window_batch* b, int mode, const bp_outputs* out) {
    if (!out) return fail(BP_ERR_INVALID, "outputs missing");
    if (mode != BP_MODE_CONJUGATE && mode != BP_MODE_JEFFREYS) return fail(BP_ERR_INVALID, "mode must be 0 or 1");
    if (out->weights || out->nu || out->w1 || out->status)
        return fail(BP_ERR_INVALID, "bp_moments_batched does not solve: use bp_conjugate_batched / bp_jeffreys_batched");
    return run_batches(h, b, out, mode, false);
}

int bp_backtest_batched(bp_handle* h, const bp_backtest_desc* d) {
    if (!h || !d) return fail(BP_ERR_INVALID, "null argument");
    if (!h->has_market) return fail(BP_ERR_STATE, "no market uploaded");
    if (!h->has_caps) return fail(BP_ERR_STATE, "the backtest loop needs market caps (comparison portfolio)");
    const int R = d->n_rebalances, N = h->N;
    if (R < 1 || !d->reb_row || !d->weights || !d->returns || !d->turnover || !d->metrics)
        return fail(BP_ERR_INVALID, "bp_backtest_desc incomplete");
    if (N > 8 * 256) return fail(BP_ERR_INVALID, "the loop kernel supports at most 2048 assets");
    if (is_device_ptr(d->reb_row)) return fail(BP_ERR_INVALID, "reb_row must be a host pointer");
    for (int s = 0; s < R; ++s) {
        const int r = d->reb_row[s];
        if (r < 1 || r >= h->D || (s > 0 && r <= d->reb_row[s - 1]))
            return fail(BP_ERR_INVALID, "reb_row must be ascending rows in [1, n_days)");
    }
    CU_TRY(cudaSetDevice(h->device));
    cudaStream_t st = h->stream;
    if (d->last_row < d->reb_row[R - 1] || d->last_row >= h->D) return fail(BP_ERR_INVALID, "last_row must lie in [reb_row[R-1], n_days)");
    const int T = d->last_row - d->reb_row[0];
    // workspace: weights, member, reb_row, returns, turnover, metrics
    auto al = [](size_t x) { return (x + 15) & ~(size_t)15; };
    const size_t b_w = al(sizeof(double) * (size_t)R * N), b_m = al((size_t)R * N), b_r = al(sizeof(int) * (size_t)R);
    const size_t b_ret = al(sizeof(double) * (size_t)std::max(T, 1)), b_to = al(sizeof(double) * (size_t)std::max(R - 1, 1));
    const size_t b_met = al(sizeof(double) * (size_t)R * 5);
    int rc = grow(h, h->ws, b_w + b_m + b_r + b_ret + b_to + b_met + 256);
    if (rc) return rc;
    unsigned char* base = h->ws.p;
    double* dw = reinterpret_cast<double*>(base);                    base += b_w;
    unsigned char* dm = base;                                          base += b_m;
    int* dr = reinterpret_cast<int*>(base);                           base += b_r;
    double* dret = reinterpret_cast<double*>(base);                   base += b_ret;
    double* dto = reinterpret_cast<double*>(base);                    base += b_to;
    double* dmet = reinterpret_cast<double*>(base);
    const double* wsrc = d->weights;
    if (!is_device_ptr(d->weights)) {
        CU_TRY(cudaMemcpyAsync(dw, d->weights, sizeof(double) * (size_t)R * N, cudaMemcpyHostToDevice, st));
        wsrc = dw;
    }
    const unsigned char* msrc = d->member;
    if (d->member && !is_device_ptr(d->member)) {
        CU_TRY(cudaMemcpyAsync(dm, d->member, (size_t)R * N, cudaMemcpyHostToDevice, st));
        msrc = dm;
    }
    CU_TRY(cudaMemcpyAsync(dr, d->reb_row, sizeof(int) * (size_t)R, cudaMemcpyHostToDevice, st));
    LoopParams lp{};
    lp.n_assets = N; lp.n_rebalances = R; lp.ldw = N;
    lp.weights = wsrc; lp.member = msrc; lp.reb_row = dr; lp.last_row = d->last_row;
    lp.prices = h->prices; lp.ld_prices = N; lp.caps = h->caps; lp.ld_caps = N; lp.rf_row = h->rf_row;
    lp.distance_scale = d->distance_scale; lp.turnover_cost_bps = d->turnover_cost_bps;
    lp.returns = dret; lp.turnover = dto; lp.metrics = dmet;
    CU_TRY(launch_backtest_loop(lp, st));
    h->launches++;
    if (T > 0 && (rc = emit_raw(h, dret, sizeof(double) * (size_t)T, d->returns))) return rc;
    if (R > 1 && (rc = emit_raw(h, dto, sizeof(double) * (size_t)(R - 1), d->turnover))) return rc;
    if ((rc = emit_raw(h, dmet, sizeof(double) * (size_t)R * 5, d->metrics))) return rc;
    CU_TRY(cudaStreamSynchronize(st));       // the staging copies of host inputs must be consumed before return
    h->need_sync = false;
    return BP_OK;
}

int bp_excess_returns(bp_handle* h, const bp_window_batch* b, double* X) {
    if (!h || !b || !X) return fail(BP_ERR_INVALID, "null argument");
    if (b->n_windows != 1) return fail(BP_ERR_INVALID, "bp_excess_returns handles one window per call");
    int rc = check_batch(plan_ctx(h), b, false, &g_err);
    if (rc) return rc;
    CU_TRY(cudaSetDevice(h->device));
    const int K = b->rolling_window - 1;
    const size_t bytes = sizeof(double) * (size_t)K * h->N;
    const bool dev = is_device_ptr(X);
    double* dst = X;
    if (!dev) {
        if ((rc = grow(h, h->stage, bytes))) return rc;
        dst = reinterpret_cast<double*>(h->stage.p);
    }
    launch_excess_returns(h->lr_d, h->ld, h->rf_row, b->day_row[0], b->span_days[0], b->rolling_window, h->N, dst, h->stream);
    h->launches++;
    CU_TRY(cudaGetLastError());
    if (!dev) {
        CU_TRY(cudaMemcpyAsync(X, dst, bytes, cudaMemcpyDeviceToHost, h->stream));
        CU_TRY(cudaStreamSynchronize(h->stream));
    }
    return BP_OK;
}

int bp_quadratic_form(bp_handle* h, int n, const double* w, const double* S, double* out) {
    if (!h || !w || !S || !out || n <= 0) return fail(BP_ERR_INVALID, "bad argument");
    CU_TRY(cudaSetDevice(h->device));
    const size_t need = sizeof(double) * ((size_t)n * n + n + 8);
    int rc = grow(h, h->stage, need);
    if (rc) return rc;
    double* dS = reinterpret_cast<double*>(h->stage.p);
    double* dw = dS + (size_t)n * n;
    double* dv = dw + n;
    CU_TRY(cudaMemcpyAsync(dS, S, sizeof(double) * (size_t)n * n, cudaMemcpyHostToDevice, h->stream));
    CU_TRY(cudaMemcpyAsync(dw, w, sizeof(double) * (size_t)n, cudaMemcpyHostToDevice, h->stream));
    launch_quadform(dS, n, dw, n, dv, 0.0, 0.0, nullptr, nullptr, h->stream);
    h->launches++;
    CU_TRY(cudaGetLastError());
    CU_TRY(cudaMemcpyAsync(out, dv, sizeof(double), cudaMemcpyDeviceToHost, h->stream));
    CU_TRY(cudaStreamSynchronize(h->stream));
    return BP_OK;
}

int bp_dense_posterior(bp_handle* h, const bp_dense_problem* in, const bp_dense_result* out) {
    if (!h || !in || !out) return fail(BP_ERR_INVALID, "null argument");
    const int N = in->n_assets;
    const bool c_only = !in->T && !in->t && !in->jeffreys;
    if (N <= 0 || (!c_only && (!in->T || !in->t))) return fail(BP_ERR_INVALID, "T and t are required");
    if (!in->jeffreys && (!in->S0 || !in->w0)) return fail(BP_ERR_INVALID, "conjugate posterior needs S0 and w0");
    if (!(in->risk_aversion != 0.0)) return fail(BP_ERR_INVALID, "risk_aversion must be non-zero");
    const bool solves = !c_only && (in->jeffreys || !in->w1);      // an injected posterior w skips the solver
    int rc = BP_OK;
    if (solves && (rc = check_solver_size(N, BP_EST_NONE))) return rc;
    CU_TRY(cudaSetDevice(h->device));
    const int ldS = round_up(N, 32), rowsS = ldS + 8, ldv = round_up(N, 16);
    const size_t NN = (size_t)N * N;
    auto al = [](size_t x) { return (x + 3) & ~(size_t)3; };      // keep every carve 32-byte aligned
    const size_t doubles = 3 * al(NN) + 4 * al(N) + 4 * al(ldv) + (size_t)rowsS * ldS + al(BP_NSCAL) + 8;
    rc = grow(h, h->ws, sizeof(double) * doubles + 64);
    if (rc) return rc;
    double* p = reinterpret_cast<double*>(h->ws.p);
    double* dT = p;            p += al(NN);
    double* dS0 = p;           p += al(NN);
    double* dS1in = p;         p += al(NN);
    double* dt = p;            p += al(N);
    double* dw0 = p;           p += al(N);
    double* dw1in = p;         p += al(N);
    double* ds0w0 = p;         p += al(N);
    double* drhs = p;          p += al(ldv);
    double* dw1 = p;           p += al(ldv);
    double* dnu = p;           p += al(ldv);
    double* dwts = p;          p += al(ldv);
    double* dscal = p;         p += al(BP_NSCAL);
    double* dS = p;            p += (size_t)rowsS * ldS;
    int* dstatus = reinterpret_cast<int*>(p);
    cudaStream_t st = h->stream;
    CU_TRY(cudaMemsetAsync(dscal, 0, sizeof(double) * BP_NSCAL, st));
    CU_TRY(cudaMemsetAsync(dstatus, 0, sizeof(int), st));
    if (!c_only) {
        CU_TRY(cudaMemcpyAsync(dT, in->T, sizeof(double) * NN, cudaMemcpyHostToDevice, st));
        CU_TRY(cudaMemcpyAsync(dt, in->t, sizeof(double) * N, cudaMemcpyHostToDevice, st));
    }
    if (!in->jeffreys) {
        CU_TRY(cudaMemcpyAsync(dS0, in->S0, sizeof(double) * NN, cudaMemcpyHostToDevice, st));
        CU_TRY(cudaMemcpyAsync(dw0, in->w0, sizeof(double) * N, cudaMemcpyHostToDevice, st));
        if (in->S1) CU_TRY(cudaMemcpyAsync(dS1in, in->S1, sizeof(double) * NN, cudaMemcpyHostToDevice, st));
        if (in->w1) CU_TRY(cudaMemcpyAsync(dw1in, in->w1, sizeof(double) * N, cudaMemcpyHostToDevice, st));
    }
    const double n1 = in->n1 ? *in->n1 : in->n0 + (double)in->rolling_window;
    DenseParams dp{};
    dp.n_assets = N; dp.ldS = ldS; dp.ldv = ldv; dp.n_window = in->rolling_window;
    dp.n0 = in->n0; dp.n1 = n1; dp.has_c = in->c != nullptr; dp.c_in = in->c ? *in->c : 0.0;
    dp.T = c_only ? nullptr : dT; dp.t = c_only ? nullptr : dt; dp.S0 = dS0; dp.w0 = dw0; dp.S1_in = (!in->jeffreys && in->S1) ? dS1in : nullptr;
    dp.s0w0 = ds0w0; dp.rhs = drhs; dp.S_out = dS; dp.scal = dscal;
    launch_dense_prep(dp, in->jeffreys != 0, st);
    h->launches++;
    CU_TRY(cudaGetLastError());
    if (c_only) {
        if (out->scalars) CU_TRY(cudaMemcpyAsync(out->scalars, dscal, sizeof(double) * BP_NSCAL, cudaMemcpyDeviceToHost, st));
        CU_TRY(cudaStreamSynchronize(st));
        return BP_OK;
    }
    const Layout L = make_layout(N, ldv, 0, false);
    if (out->S1) {
        if ((rc = emit_dense(h, dS, L, 1, true, out->S1))) return rc;
        if (h->need_sync) { CU_TRY(cudaStreamSynchronize(st)); h->need_sync = false; }
    }
    const double inv_gamma = 1.0 / in->risk_aversion;
    if (!in->jeffreys && in->w1) {
        // injected posterior w: v1 = w1'S1w1 (:574), nu (:572-575), weights (:836)
        launch_quadform(dS, ldS, dw1in, N, dscal + BP_SCAL_V1, n1, inv_gamma, dnu, dwts, st);
        h->launches++;
        CU_TRY(cudaMemcpyAsync(dw1, dw1in, sizeof(double) * N, cudaMemcpyDeviceToDevice, st));
    } else {
        Chunk c{};
        c.S = dS; c.rhs = drhs; c.scal = dscal; c.w1 = dw1; c.nu = dnu; c.weights = dwts; c.status = dstatus;
        if ((rc = solve_windows(h, c, L, 1, 1, in->jeffreys ? BP_MODE_JEFFREYS : BP_MODE_CONJUGATE, BP_EST_NONE, 0, inv_gamma)))
            return rc;
    }
    CU_TRY(cudaGetLastError());
    if (out->scalars) CU_TRY(cudaMemcpyAsync(out->scalars, dscal, sizeof(double) * BP_NSCAL, cudaMemcpyDeviceToHost, st));
    if (out->w1) CU_TRY(cudaMemcpyAsync(out->w1, dw1, sizeof(double) * N, cudaMemcpyDeviceToHost, st));
    if (out->nu) CU_TRY(cudaMemcpyAsync(out->nu, dnu, sizeof(double) * N, cudaMemcpyDeviceToHost, st));
    if (out->weights) CU_TRY(cudaMemcpyAsync(out->weights, dwts, sizeof(double) * N, cudaMemcpyDeviceToHost, st));
    if (out->status) CU_TRY(cudaMemcpyAsync(out->status, dstatus, sizeof(int), cudaMemcpyDeviceToHost, st));
    CU_TRY(cudaStreamSynchronize(st));
    return BP_OK;
}

int bp_solve_batched(bp_handle* h, const bp_solve_desc* d, const bp_outputs* out) {
    if (!h || !d || !out) return fail(BP_ERR_INVALID, "null argument");
    const int W = d->n_windows, N = d->n_assets;
    if (W <= 0 || N <= 0) return fail(BP_ERR_INVALID, "need n_windows > 0 and n_assets > 0");
    if (!d->S || !d->rhs) return fail(BP_ERR_INVALID, "S and rhs are required");
    if (d->estimator != BP_EST_NONE && d->estimator != BP_EST_JORION)
        return fail(BP_ERR_INVALID, "estimator must be 0 or BP_ESTIMATOR_JORION");
    const bool jorion = d->estimator == BP_EST_JORION;
    const int mode = (d->jeffreys || jorion) ? BP_MODE_JEFFREYS : BP_MODE_CONJUGATE;
    if (mode == BP_MODE_CONJUGATE && !d->n1) return fail(BP_ERR_INVALID, "the conjugate scaling needs n1");
    if (jorion && d->n_returns - N - 2 <= 0) return fail(BP_ERR_INVALID, "Jorion needs n_returns - N - 2 > 0 (:879)");
    if (!(d->risk_aversion != 0.0)) return fail(BP_ERR_INVALID, "risk_aversion must be non-zero");
    if (out->T || out->S0 || out->S1 || out->t || out->w0 || out->rhs)
        return fail(BP_ERR_INVALID, "bp_solve_batched returns w1, nu, weights, scalars and status only");
    int rc = check_solver_size(N, d->estimator);
    if (rc) return rc;
    CU_TRY(cudaSetDevice(h->device));
    // the layout of bp_dense_posterior for W windows
    const Layout L = make_layout(N, round_up(N, 16), 0, false);
    const int Wc = (int)std::min<size_t>((size_t)W, std::max<size_t>(1, h->ws_limit / L.per_window));
    if ((rc = grow(h, h->ws, (size_t)Wc * L.per_window + 256))) return rc;
    const Chunk c = carve(h->ws.p, L, Wc);
    cudaStream_t st = h->stream;
    for (int w0 = 0; w0 < W; w0 += Wc) {
        const int wc = std::min(Wc, W - w0);
        const size_t NN = (size_t)N * N;
        // only the N x N entries of each window: the padding rows and columns keep whatever the workspace held
        for (int k = 0; k < wc; ++k)
            CU_TRY(cudaMemcpy2DAsync(c.S + (size_t)k * L.win_stride, sizeof(double) * L.ldS, d->S + (size_t)(w0 + k) * NN,
                                     sizeof(double) * N, sizeof(double) * N, N, cudaMemcpyHostToDevice, st));
        CU_TRY(cudaMemcpy2DAsync(c.rhs, sizeof(double) * L.ldv, d->rhs + (size_t)w0 * N, sizeof(double) * N,
                                 sizeof(double) * N, wc, cudaMemcpyHostToDevice, st));
        CU_TRY(cudaMemsetAsync(c.scal, 0, sizeof(double) * BP_NSCAL * (size_t)wc, st));
        if (mode == BP_MODE_CONJUGATE)
            CU_TRY(cudaMemcpy2DAsync(c.scal + BP_SCAL_N1, sizeof(double) * BP_NSCAL, d->n1 + w0, sizeof(double), sizeof(double),
                                     wc, cudaMemcpyHostToDevice, st));
        if ((rc = solve_windows(h, c, L, wc, 1, mode, d->estimator, d->n_returns, 1.0 / d->risk_aversion))) return rc;
        // (t, w0 and rhs are not outputs of this call: the checks above rejected them)
        if ((rc = emit_chunk(h, c, L, out, w0, wc, W, true, false))) return rc;
    }
    return finish(h);
}

}  // extern "C"
