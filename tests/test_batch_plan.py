"""CPU tests of the window-batch planner (csrc/batch_plan.cu): the descriptor image of every planned window covers
its daily and intraday return rows exactly once, every block / range / triple id is in range, and invalid batches
are rejected with the library's messages.  The planner is host code only; it is compiled here with g++."""
import ctypes as C
import dataclasses
import os
import shutil
import subprocess

import numpy as np
import pytest

from incorporating_different_sources_b200._lib import WindowBatchDesc
from incorporating_different_sources_b200.synthetic import generate_market
from incorporating_different_sources_b200.windows import plan_daily_windows

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "incorporating_different_sources_b200", "csrc")
GDI, PHI = 20, 10          # GRAM_DESC_INTS, GRAM_PHASE_INTS

CTX = ["has_market", "N", "ld", "D", "Rw", "n_mcm", "R", "hf_extra_rows", "has_caps", "has_mcm_w", "ws_limit",
       "reuse_min_windows", "presum_min_days", "stride", "stacked", "cond_estimate", "chain_group", "chain_max",
       "chain_smem_fits", "hf_pending", "n_seg", "seg_waited"]
CALL = ["mode", "solve", "estimator", "T", "S0", "S1"]
LAYOUT = ["N", "ldv", "ldS", "rowsS", "win_stride", "y_stride", "mv_stride", "per_window"]
INFO = (["ints", "off_gram"] + [f"off_blocks{ph}{l}" for ph in (0, 1) for l in (0, 1)] + ["off_ranges0", "off_ranges1",
        "off_triples", "off_starts", "off_vids"] + [f"nb{ph}{l}" for ph in (0, 1) for l in (0, 1)] +
        [f"blk{ph}{l}" for ph in (0, 1) for l in (0, 1)] + [f"bmin{ph}{l}" for ph in (0, 1) for l in (0, 1)] +
        ["inner", "chunk", "presum", "band_ok", "nranges0", "nranges1", "nfull", "max_m", "stride"])

SHIM = r"""
#include "batch_plan.h"
#include <cstdio>
using namespace bp;

static PlanCtx ctx_of(const long long* c) {
    PlanCtx x;
    x.has_market = c[0] != 0;
    x.N = (int)c[1]; x.ld = (int)c[2]; x.D = (int)c[3]; x.Rw = (int)c[4]; x.n_mcm = (int)c[5];
    x.R = c[6];
    x.hf_extra_rows = c[7];
    x.has_caps = c[8] != 0;
    x.has_mcm_w = c[9] != 0;
    x.ws_limit = (size_t)c[10];
    x.reuse_min_windows = (int)c[11];
    x.presum_min_days = (int)c[12];
    x.stride = (int)c[13];
    x.stacked = c[14] != 0;
    x.cond_estimate = c[15] != 0;
    x.chain_group = (int)c[16];
    x.chain_max = (int)c[17];
    x.chain_smem_fits = c[18] != 0;
    x.hf_pending = c[19] != 0;
    x.n_seg = (int)c[20];
    x.seg_waited = (int)c[21];
    return x;
}

static CallDesc call_of(const int* c) {
    CallDesc x;
    x.mode = c[0];
    x.solve = c[1] != 0;
    x.estimator = c[2];
    x.T = c[3] != 0; x.S0 = c[4] != 0; x.S1 = c[5] != 0;
    return x;
}

static void put_layout(const Layout& L, long long* o) {
    o[0] = L.N; o[1] = L.ldv; o[2] = L.ldS; o[3] = L.rowsS; o[4] = L.win_stride; o[5] = L.y_stride; o[6] = L.mv_stride;
    o[7] = (long long)L.per_window;
}

extern "C" int shim_check(const long long* c, const bp_window_batch* b, int need_hf, char* msg, int cap) {
    std::string err;
    const int rc = check_batch(ctx_of(c), b, need_hf != 0, &err);
    snprintf(msg, cap, "%s", err.c_str());
    return rc;
}

extern "C" int shim_check_call(const long long* c, const bp_window_batch* b, const int* call, char* msg, int cap) {
    std::string err;
    const int rc = check_call(ctx_of(c), b, call_of(call), &err);
    snprintf(msg, cap, "%s", err.c_str());
    return rc;
}

extern "C" int shim_chain_group(const long long* c, const bp_window_batch* b, const int* call) {
    return plan_chain_group(ctx_of(c), b, call_of(call));
}

// the route of a batch planned with stride G: o = pipelined, Wc, hf_wait_rows, layout (LAYOUT)
extern "C" int shim_route(const long long* c, const bp_window_batch* b, const int* call, int G, long long* o, char* msg, int cap) {
    PlanCtx ctx = ctx_of(c);
    ctx.stride = G >= 2 ? G : 1;
    BatchPlan P;
    Route r;
    std::string err;
    int rc = plan_batch(ctx, b, call[0] == BP_MODE_CONJUGATE, &P, &err);
    if (!rc) rc = plan_route(ctx, P, b, call_of(call), G, &r, &err);
    snprintf(msg, cap, "%s", err.c_str());
    if (rc) return rc;
    o[0] = r.pipelined; o[1] = r.Wc; o[2] = r.hf_wait_rows;
    put_layout(r.L, o + 3);
    return 0;
}

extern "C" void shim_layout(int N, int ld, int max_m, int with_mv, long long* o) { put_layout(make_layout(N, ld, max_m, with_mv != 0), o); }

// the layout bp_solve_batched used to write out by hand
extern "C" void shim_solve_layout_by_hand(int N, long long* o) {
    Layout L{};
    L.N = N;
    L.ldv = round_up(N, 16);
    L.ldS = round_up(N, 32);
    L.rowsS = L.ldS + 8;
    L.win_stride = (long long)L.rowsS * L.ldS;
    L.y_stride = 2;
    L.mv_stride = 0;
    L.per_window = sizeof(double) * ((size_t)L.win_stride + 9 * (size_t)L.ldv + BP_NSCAL + (size_t)L.y_stride) + 16;
    put_layout(L, o);
}

// plan fields in the order of INFO; the image is written when it fits `cap` ints
extern "C" int shim_plan(const long long* c, const bp_window_batch* b, int need_hf, long long* o, int* image, long long cap) {
    BatchPlan P;
    std::string err;
    const int rc = plan_batch(ctx_of(c), b, need_hf != 0, &P, &err);
    if (rc) return rc;
    *o++ = (long long)P.ints; *o++ = (long long)P.off_gram;
    for (int ph = 0; ph < 2; ++ph) for (int l = 0; l < 2; ++l) *o++ = (long long)P.off_blocks[ph][l];
    *o++ = (long long)P.off_ranges[0]; *o++ = (long long)P.off_ranges[1];
    *o++ = (long long)P.off_triples; *o++ = (long long)P.off_starts; *o++ = (long long)P.off_vids;
    for (int ph = 0; ph < 2; ++ph) for (int l = 0; l < 2; ++l) *o++ = P.phase[ph].nb[l];
    for (int ph = 0; ph < 2; ++ph) for (int l = 0; l < 2; ++l) *o++ = P.phase[ph].blk[l];
    for (int ph = 0; ph < 2; ++ph) for (int l = 0; l < 2; ++l) *o++ = P.phase[ph].bmin[l];
    *o++ = P.phase[0].inner; *o++ = P.phase[0].chunk; *o++ = P.presum; *o++ = P.band_ok;
    *o++ = P.nranges[0]; *o++ = P.nranges[1]; *o++ = P.nfull; *o++ = P.max_m; *o++ = P.stride;
    if ((long long)P.ints <= cap) write_batch(P, b, image);
    return 0;
}
"""


@pytest.fixture(scope="module")
def shim(tmp_path_factory):
    gxx = shutil.which("g++")
    if gxx is None:
        pytest.skip("g++ not available")
    d = tmp_path_factory.mktemp("batch_plan")
    src = d / "shim.cpp"
    src.write_text(SHIM)
    so = d / "libbatch_plan_shim.so"
    cmd = [gxx, "-O1", "-std=c++17", "-shared", "-fPIC", "-x", "c++", os.path.join(CSRC, "batch_plan.cu"), str(src),
           "-I/usr/local/cuda/include", "-I", CSRC, "-I", os.path.join(ROOT, "include"), "-o", str(so)]
    r = subprocess.run(cmd, capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    lib = C.CDLL(str(so))
    lib.shim_check.argtypes = [C.c_void_p, C.POINTER(WindowBatchDesc), C.c_int, C.c_char_p, C.c_int]
    lib.shim_plan.argtypes = [C.c_void_p, C.POINTER(WindowBatchDesc), C.c_int, C.c_void_p, C.c_void_p, C.c_longlong]
    lib.shim_check_call.argtypes = [C.c_void_p, C.POINTER(WindowBatchDesc), C.c_void_p, C.c_char_p, C.c_int]
    lib.shim_chain_group.argtypes = [C.c_void_p, C.POINTER(WindowBatchDesc), C.c_void_p]
    lib.shim_route.argtypes = [C.c_void_p, C.POINTER(WindowBatchDesc), C.c_void_p, C.c_int, C.c_void_p, C.c_char_p, C.c_int]
    lib.shim_layout.argtypes = [C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p]
    lib.shim_solve_layout_by_hand.argtypes = [C.c_int, C.c_void_p]
    return lib


class Case:
    """A batch of the synthetic market with the handle state the planner reads."""

    def __init__(self, mkt, batch, need_hf=True, **ctx):
        self.batch, self.need_hf = batch, need_hf
        n_assets = mkt.prices.shape[1]
        R = len(mkt.hf_ts)
        self.ctx = dict(has_market=1, N=n_assets, ld=(n_assets + 15) // 16 * 16, D=mkt.n_days, Rw=0, n_mcm=2, R=R,
                        hf_extra_rows=R // 8 + 64, has_caps=1, has_mcm_w=0, ws_limit=24 << 30, reuse_min_windows=32,
                        presum_min_days=8, stride=1, stacked=0, cond_estimate=0, chain_group=8, chain_max=8,
                        chain_smem_fits=1, hf_pending=0, n_seg=0, seg_waited=0)
        self.ctx.update(ctx)
        self.keep = []
        d = WindowBatchDesc()
        d.n_windows = len(batch.day_row)
        d.rolling_window = int(batch.rolling_window)
        for name in ("day_row", "span_days") + (("hf_lo", "hf_hi") if need_hf else ()):
            a = np.ascontiguousarray(getattr(batch, name), dtype=np.int32)
            self.keep.append(a)
            setattr(d, name, a.ctypes.data)
        d.mcm_index = int(batch.mcm_index)
        d.prior_weights = int(batch.prior_weights)
        d.mcm_rows = int(batch.mcm_rows)
        d.risk_aversion = 2.0
        self.desc = d

    def _ctx(self):
        c = np.array([self.ctx[k] for k in CTX], dtype=np.int64)
        self.keep.append(c)
        return c.ctypes.data

    def check(self, lib):
        msg = C.create_string_buffer(1024)
        rc = lib.shim_check(self._ctx(), C.byref(self.desc), int(self.need_hf), msg, len(msg))
        return rc, msg.value.decode()

    def plan(self, lib):
        assert self.check(lib) == (0, "")
        info = np.zeros(len(INFO), dtype=np.int64)
        assert lib.shim_plan(self._ctx(), C.byref(self.desc), int(self.need_hf), info.ctypes.data, None, 0) == 0
        img = np.zeros(int(info[0]), dtype=np.int32)
        assert lib.shim_plan(self._ctx(), C.byref(self.desc), int(self.need_hf), info.ctypes.data, img.ctypes.data,
                             img.size) == 0
        return dict(zip(INFO, info.tolist())), img

    def _call(self, call):
        c = np.array([call.get(k, 0) for k in CALL], dtype=np.int32)
        self.keep.append(c)
        return c.ctypes.data

    def check_call(self, lib, **call):
        msg = C.create_string_buffer(1024)
        rc = lib.shim_check_call(self._ctx(), C.byref(self.desc), self._call(call), msg, len(msg))
        return rc, msg.value.decode()

    def chain_group(self, lib, **call):
        assert self.check(lib) == (0, "")
        return lib.shim_chain_group(self._ctx(), C.byref(self.desc), self._call(call))

    def route(self, lib, G=0, **call):
        """(rc, message, dict with pipelined, Wc, hf_wait_rows and the layout's fields)"""
        assert self.check(lib) == (0, "")
        o = np.zeros(3 + len(LAYOUT), dtype=np.int64)
        msg = C.create_string_buffer(1024)
        rc = lib.shim_route(self._ctx(), C.byref(self.desc), self._call(call), G, o.ctypes.data, msg, len(msg))
        return rc, msg.value.decode(), dict(zip(["pipelined", "Wc", "hf_wait_rows"] + LAYOUT, o.tolist()))

    def set_rows(self, name, rows):
        a = np.ascontiguousarray(rows, dtype=np.int32)
        self.keep.append(a)
        setattr(self.desc, name, a.ctypes.data)


def _spec(n):
    return dict(weighting_strategy="conjugate_hf_vix_vw", size=8, risk_aversion=2, rolling_window=n,
                rolling_window_frequency="daily", mcm_scaling=3)


def _mkt(n_days, **kw):
    return generate_market(8, n_days, seed=11, **kw)


def _daily(mkt, d_idx, look, n=252, **ctx):
    return Case(mkt, plan_daily_windows(_spec(n), mkt.dates, d_idx, mkt.hf_ts, hf_lookback_days=look), **ctx)


def _irregular(look):
    n, W, nwin = 24, 48, 60          # as test_gpu_configs.test_irregular_intraday_calendar_day_blocks
    base = generate_market(n, 40 + nwin + W, seed=77, bars_per_day=26)
    rng = np.random.default_rng(5)
    keep = np.ones(len(base.hf_ts), dtype=bool)
    B = 26
    for day in rng.choice(base.n_days, size=12, replace=False):
        keep[day * B + 13: (day + 1) * B] = False
    keep[rng.choice(len(keep), size=60, replace=False)] = False
    keep[(base.n_days - 20) * B + 9: (base.n_days - 19) * B] = False
    mkt = dataclasses.replace(base, hf_ts=base.hf_ts[keep], hf_prices=np.ascontiguousarray(base.hf_prices[keep]))
    d_idx = list(range(mkt.n_days - W, mkt.n_days))
    return Case(mkt, plan_daily_windows(_spec(nwin), mkt.dates, d_idx, mkt.hf_ts, hf_lookback_days=look))


def _jeffreys_chain():
    mkt = _mkt(1010 + 64, bars_per_day=2)
    batch = plan_daily_windows(dict(_spec(1008), weighting_strategy="jeffreys"), mkt.dates, range(1010, 1074),
                               need_hf=False)
    return Case(mkt, batch, need_hf=False, stride=8)


CASES = {
    "consecutive_7d": lambda: _daily(_mkt(330), range(260, 320), 7),
    "every_third_7d": lambda: _daily(_mkt(400), range(260, 380, 3), 7),
    "random_7d": lambda: _daily(_mkt(400), np.sort(np.random.default_rng(3).choice(np.arange(260, 400), 48, replace=False)), 7),
    "lookback_252d": lambda: _daily(_mkt(330), range(260, 320), 252),
    "irregular_7d": lambda: _irregular(7),
    "irregular_31d": lambda: _irregular(31),
    "below_reuse_min": lambda: _daily(_mkt(330), range(260, 280), 7),
    "jeffreys_chain": _jeffreys_chain,
    "ws_limit_gives_up": lambda: _daily(_mkt(330), range(260, 320), 7, ws_limit=12 << 20),
}


def _rows_once(parts, lo, hi):
    """parts: list of row arrays; True when together they cover [lo, hi) exactly once."""
    rows = np.concatenate([np.asarray(p, dtype=np.int64) for p in parts]) if parts else np.zeros(0, np.int64)
    return np.array_equal(np.sort(rows), np.arange(lo, hi))


def _span(r0, n):
    return np.arange(r0, r0 + n)


def _block_rows(img, P, ph, l, k):
    assert 0 <= k < P[f"nb{ph}{l}"]
    d = img[P[f"off_blocks{ph}{l}"] + k * GDI + ph * PHI:][:PHI]
    return _span(d[0], d[1])


def _check_daily(img, P, dr, n, d):
    parts = [_span(d[0], d[1]), _span(d[2], d[3])]
    if d[5]:
        assert d[5] == 1 and not d[6:].any() and 0 <= d[4] < P["nfull"]
        triple = img[P["off_triples"] + 3 * d[4]:][:3]
        for level, rid in zip((0, 1, 1), triple):
            if rid < 0:
                continue
            assert rid < P[f"nranges{level}"]
            lo, hi = img[P[f"off_ranges{level}"] + 2 * rid:][:2]
            assert 0 <= lo < hi <= P[f"nb1{level}"]
            parts += [_block_rows(img, P, 1, level, k) for k in range(lo, hi)]
    assert _rows_once(parts, dr - n + 2, dr + 1)


def _check_intraday(img, P, case, lo, hi, d, vid):
    R, nb0 = case.ctx["R"], P["nb00"]
    if not P["inner"]:
        parts = [_span(d[0], d[1]), _span(d[2], d[3])]
        for (b0, cnt), l in zip(d[4:10].reshape(3, 2), (0, 1, 1)):
            parts += [_block_rows(img, P, 0, l, k) for k in range(b0, b0 + cnt)]
        assert _rows_once(parts, lo + 1, hi)
        return
    starts = img[P["off_starts"]:][:nb0 + 1]
    assert np.all(np.diff(starts) > 0)
    inner = lambda k: np.arange(starts[k] + 1, starts[k + 1])      # noqa: E731
    full = lambda k: np.arange(starts[k], starts[k + 1])           # noqa: E731
    for k in range(nb0):
        assert np.array_equal(_block_rows(img, P, 0, 0, k), inner(k))
    if not P["presum"]:
        assert d[2] == d[3] == 0 and not d[6:10].any()
        assert 0 <= d[4] and d[4] + d[5] <= nb0
        assert R <= d[0] and d[0] + d[1] <= R + case.ctx["hf_extra_rows"]
        parts = [inner(k) for k in range(d[4], d[4] + d[5])]
        parts.append(starts[np.arange(d[0], d[0] + d[1]) - R])     # gathered row R+k is return row starts[k]
        assert _rows_once(parts, lo + 1, hi)
        return
    C_ = P["chunk"]
    ids = [i for i in vid if i >= 0]
    assert 1 <= len(ids) <= 3 and vid[0] >= 0
    assert not d[:4].any()
    for k in range(3):
        assert (d[4 + 2 * k], d[5 + 2 * k]) == ((vid[k], 1) if vid[k] >= 0 else (0, 0))
    parts = []
    for i in ids:
        assert nb0 <= i < 3 * nb0
        if i < 2 * nb0:                # suffix'[f]: inner[f] + FD[f+1 .. end of f's chunk]
            f = i - nb0
            parts += [inner(f)] + [full(k) for k in range(f + 1, min((f // C_ + 1) * C_, nb0))]
        else:                          # prefix[b]: FD[start of b's chunk .. b]
            b = i - 2 * nb0
            parts += [full(k) for k in range(b // C_ * C_, b + 1)]
    assert _rows_once(parts, lo + 1, hi)


@pytest.mark.parametrize("name", list(CASES))
def test_plan_covers_every_window_row_once(shim, name):
    case = CASES[name]()
    P, img = case.plan(shim)
    b = case.batch
    W, n = len(b.day_row), int(b.rolling_window)
    assert np.array_equal(img[:W], b.day_row) and np.array_equal(img[W:2 * W], b.span_days)
    expect = {
        "consecutive_7d": dict(inner=1, blk10=64, blk11=16, band_ok=1, presum=0),
        "every_third_7d": dict(inner=0, blk00=64, blk01=16, band_ok=0),
        "lookback_252d": dict(inner=1, presum=1),
        "below_reuse_min": dict(nb00=0, nb01=0, nb10=0, nb11=0),
        "jeffreys_chain": dict(blk10=128, blk11=32, stride=8),
        "ws_limit_gives_up": dict(nb00=0, nb01=0, inner=0, blk10=64),
    }.get(name, {})
    assert {k: P[k] for k in expect} == expect
    if name.startswith("irregular"):
        assert P["inner"] == 1 and P["presum"] == (name == "irregular_31d")
    if name == "ws_limit_gives_up":
        assert P["nb10"] > 0          # the daily phase keeps its blocks
    for w in range(0, W, P["stride"]):
        gd = img[P["off_gram"] + w * GDI:][:GDI]
        _check_daily(img, P, int(b.day_row[w]), n, gd[PHI:])
        if case.need_hf:
            lo, hi = int(b.hf_lo[w]), int(b.hf_hi[w])
            assert img[3 * W + w] == lo + 1 and img[4 * W + w] == hi - lo - 1
            vid = img[P["off_vids"] + 3 * w:][:3] if P["presum"] else None
            _check_intraday(img, P, case, lo, hi, gd[:PHI], vid)
    if case.need_hf:
        assert P["max_m"] == int((b.hf_hi - b.hf_lo).max()) - 1


@pytest.mark.parametrize("field, value, message", [
    ("day_row", 5, "window 3: day_row 5 needs 251 prior price rows inside [0,330)"),
    ("hf_hi", None, "window 3: intraday rows [{lo},{hi}) give 1 returns (need >= 2, rows < {R})"),
    ("span_days", 0, "window 3: span_days must be positive"),
])
def test_invalid_batch_is_rejected(shim, field, value, message):
    case = _daily(_mkt(330), range(260, 320), 7)
    b = case.batch
    arr = np.array(getattr(b, field), dtype=np.int32)
    if field == "hf_hi":
        value = int(b.hf_lo[3]) + 2
    arr[3] = value
    case = Case(_mkt(330), dataclasses.replace(b, **{field: arr}))
    rc, msg = case.check(shim)
    assert rc == 1          # BP_ERR_INVALID
    assert msg == message.format(lo=int(b.hf_lo[3]), hi=value, R=case.ctx["R"])


JEFF = dict(mode=1, solve=1)          # bp_jeffreys_batched
CONJ = dict(mode=0, solve=1)          # bp_conjugate_batched


def _layout(lib, N, ld, max_m=0, with_mv=0):
    o = np.zeros(len(LAYOUT), dtype=np.int64)
    lib.shim_layout(N, ld, max_m, with_mv, o.ctypes.data)
    return dict(zip(LAYOUT, o.tolist()))


def test_solve_layout_is_make_layout(shim):
    """bp_solve_batched and bp_dense_posterior take make_layout(N, round_up(N, 16), 0, false): field by field the
    layout bp_solve_batched wrote out by hand."""
    for N in range(1, 1100):
        o = np.zeros(len(LAYOUT), dtype=np.int64)
        shim.shim_solve_layout_by_hand(N, o.ctypes.data)
        assert _layout(shim, N, (N + 15) // 16 * 16) == dict(zip(LAYOUT, o.tolist())), N


def _chain_case():
    case = _jeffreys_chain()
    case.ctx["stride"] = 1
    return case


def test_chain_group_taken(shim):
    case = _chain_case()
    assert case.chain_group(shim, **JEFF) == 8
    assert case.chain_group(shim, estimator=1, **JEFF) == 8          # Jorion chains too
    case.ctx["chain_group"] = 4
    assert case.chain_group(shim, **JEFF) == 4


@pytest.mark.parametrize("term", ["cond_estimate", "mode", "estimator", "solve", "T", "S0", "S1", "resampled", "stacked",
                                  "chain_group", "n_windows", "day_row", "smem", "workspace", "rank_margin"])
def test_chain_group_refused_by_each_term(shim, term):
    """Flipping any one term of the chain condition alone falls back to factorising every window (G = 0)."""
    case = _chain_case()
    call = dict(JEFF)
    W, n = case.desc.n_windows, case.desc.rolling_window
    per_window = _layout(shim, case.ctx["N"], case.ctx["ld"])["per_window"]
    if term in ("cond_estimate", "stacked"):
        case.ctx[term] = 1
    elif term == "mode":
        call["mode"] = 0
    elif term == "estimator":
        call["estimator"] = 2             # shrinkage
    elif term == "solve":
        call["solve"] = 0
    elif term in ("T", "S0", "S1"):
        call[term] = 1
    elif term == "resampled":             # weekly rows: row r of the resampled rows stands in for daily row r here
        case.desc.resampled = 1
        case.ctx["Rw"] = case.ctx["D"]
        case.set_rows("extra_row", case.batch.day_row)
        case.set_rows("caps_row", case.batch.day_row)
    elif term == "chain_group":
        case.ctx["chain_group"] = 1
    elif term == "n_windows":
        assert case.chain_group(shim, **call) == 8
        case.desc.n_windows = 2 * 8 - 1
    elif term == "day_row":
        rows = np.array(case.batch.day_row, dtype=np.int32)
        rows[:W // 2] -= 1                # one gap in the trade dates
        case.set_rows("day_row", rows)
    elif term == "smem":
        case.ctx["chain_smem_fits"] = 0
    elif term == "workspace":
        case.ctx["ws_limit"] = W * per_window
        assert case.chain_group(shim, **call) == 8
        case.ctx["ws_limit"] = W * per_window - 1
    elif term == "rank_margin":            # rolling_window - 1 < N + 2G + 8
        for N, G in ((n - 1 - 24, 8), (n - 1 - 23, 0)):
            case.ctx.update(N=N, ld=(N + 15) // 16 * 16)
            assert case.chain_group(shim, **call) == G, N
        return
    assert case.chain_group(shim, **call) == 0


def _pipe_case(**ctx):
    return _daily(_mkt(330), range(260, 320), 7, hf_pending=1, n_seg=4, seg_waited=1, **ctx)


def test_pipelined_route(shim):
    case = _pipe_case()
    rc, msg, r = case.route(shim, **CONJ)
    assert (rc, msg) == (0, "")
    assert r["pipelined"] == 1 and r["Wc"] == case.desc.n_windows and r["hf_wait_rows"] == 0
    rc, _, r = case.route(shim, S1=1, **CONJ)                 # S1 leaves every segment's windows on the way
    assert rc == 0 and r["pipelined"] == 1


@pytest.mark.parametrize("term", ["mode", "hf_pending", "n_seg", "seg_waited", "solve", "T", "S0", "chunked", "presum"])
def test_pipelined_refused_by_each_term(shim, term):
    call = dict(CONJ)
    case = _pipe_case()
    if term == "mode":
        case = Case(_mkt(330), case.batch, need_hf=False, **{k: case.ctx[k] for k in ("hf_pending", "n_seg", "seg_waited")})
        call["mode"] = 1
    elif term == "hf_pending":
        case.ctx["hf_pending"] = 0
    elif term == "n_seg":
        case.ctx.update(n_seg=1, seg_waited=0)
    elif term == "seg_waited":
        case.ctx["seg_waited"] = 4
    elif term in ("solve",):
        call["solve"] = 0
    elif term in ("T", "S0"):
        call[term] = 1
    elif term == "chunked":
        per_window = case.route(shim, **call)[2]["per_window"]
        case.ctx["ws_limit"] = case.desc.n_windows * per_window - 1
    elif term == "presum":
        case = _daily(_mkt(330), range(260, 320), 252, hf_pending=1, n_seg=4, seg_waited=1)
        assert case.plan(shim)[0]["presum"] == 1
    rc, msg, r = case.route(shim, **call)
    assert (rc, msg) == (0, "")
    assert r["pipelined"] == 0
    # a conjugate batch that is not pipelined waits for the intraday rows it reads first
    assert r["hf_wait_rows"] == (int(np.max(case.batch.hf_hi)) if call["mode"] == 0 else 0)


def test_wait_rows_are_the_last_row_read(shim):
    """Windows out of date order: the batch waits for the largest hf_hi, not the last window's."""
    case = _daily(_mkt(400), np.sort(np.random.default_rng(3).choice(np.arange(260, 400), 48, replace=False)), 7)
    hi = np.array(case.batch.hf_hi, dtype=np.int32)
    hi_max = int(hi.max())
    hi = np.ascontiguousarray(hi[::-1])
    case.set_rows("hf_hi", hi)
    case.set_rows("hf_lo", np.ascontiguousarray(np.array(case.batch.hf_lo, dtype=np.int32)[::-1]))
    case.set_rows("day_row", np.ascontiguousarray(np.array(case.batch.day_row, dtype=np.int32)[::-1]))
    case.set_rows("span_days", np.ascontiguousarray(np.array(case.batch.span_days, dtype=np.int32)[::-1]))
    rc, _, r = case.route(shim, **CONJ)
    assert rc == 0 and r["pipelined"] == 0 and r["hf_wait_rows"] == hi_max and hi[-1] < hi_max
    rc, _, r = case.route(shim, mode=0)                       # bp_hf_cov_batched / bp_moments_batched
    assert rc == 0 and r["hf_wait_rows"] == hi_max


def test_chunk_size_at_the_workspace_limit(shim):
    case = _daily(_mkt(330), range(260, 320), 7)
    W = case.desc.n_windows
    pw = case.route(shim, **CONJ)[2]["per_window"]
    assert pw == _layout(shim, case.ctx["N"], case.ctx["ld"], int(np.max(case.batch.hf_hi - case.batch.hf_lo)) - 1)["per_window"]
    for limit, Wc in ((10 * pw, 10), (10 * pw - 1, 9), (11 * pw, 11), (W * pw, W), (W * pw - 1, W - 1),
                      ((W + 1) * pw, W), (pw - 1, 1)):
        case.ctx["ws_limit"] = limit
        rc, msg, r = case.route(shim, **CONJ)
        assert (rc, msg, r["Wc"]) == (0, "", Wc), limit


def test_chained_batch_fits_one_chunk(shim):
    """The chain group is only taken when the whole batch fits one workspace chunk, so the route's internal check that
    a chained batch is not chunked holds at the limit."""
    case = _chain_case()
    W = case.desc.n_windows
    pw = _layout(shim, case.ctx["N"], case.ctx["ld"])["per_window"]
    for limit in (W * pw, W * pw - 1):
        case.ctx["ws_limit"] = limit
        G = case.chain_group(shim, **JEFF)
        rc, msg, r = case.route(shim, G=G, **JEFF)
        assert (rc, msg) == (0, "") and (G, r["Wc"]) == ((8, W) if limit == W * pw else (0, W - 1))
        assert r["per_window"] == pw and r["hf_wait_rows"] == 0 and r["pipelined"] == 0
    case.ctx["ws_limit"] = W * pw - 1                          # a chain group the planner would not give
    rc, msg, _ = case.route(shim, G=8, **JEFF)
    assert (rc, msg) == (4, "internal: chained batch does not fit one workspace chunk")      # BP_ERR_STATE


@pytest.mark.parametrize("call, risk_aversion, ok", [
    (CONJ, 0.0, False),
    (dict(mode=1, solve=1, estimator=1), 0.0, False),          # Jorion
    (dict(mode=1, solve=1, estimator=2), 0.0, False),          # shrinkage
    (JEFF, 0.0, True),                                         # a plain Jeffreys call never reads it
    (dict(mode=0), 0.0, True),                                 # moments only
    (CONJ, -3.0, True),
])
def test_risk_aversion_check(shim, call, risk_aversion, ok):
    case = _daily(_mkt(330), range(260, 320), 7)
    case.desc.risk_aversion = risk_aversion
    assert case.check_call(shim, **call) == ((0, "") if ok else (1, "risk_aversion must be non-zero"))


def test_jorion_needs_more_returns_than_assets(shim):
    case = _chain_case()
    n = case.desc.rolling_window
    for N, ok in ((n - 4, True), (n - 3, False), (n + 10, False)):
        case.ctx["N"] = N
        expect = (0, "") if ok else (1, "Jorion needs T - N - 2 > 0 (T = rolling_window - 1 returns, :879)")
        assert case.check_call(shim, estimator=1, **JEFF) == expect, N
        assert case.check_call(shim, estimator=2, **JEFF) == (0, "")
