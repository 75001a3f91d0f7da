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
       "reuse_min_windows", "presum_min_days", "stride"]
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
    return x;
}

extern "C" int shim_check(const long long* c, const bp_window_batch* b, int need_hf, char* msg, int cap) {
    std::string err;
    const int rc = check_batch(ctx_of(c), b, need_hf != 0, &err);
    snprintf(msg, cap, "%s", err.c_str());
    return rc;
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
    return lib


class Case:
    """A batch of the synthetic market with the handle state the planner reads."""

    def __init__(self, mkt, batch, need_hf=True, **ctx):
        self.batch, self.need_hf = batch, need_hf
        n_assets = mkt.prices.shape[1]
        R = len(mkt.hf_ts)
        self.ctx = dict(has_market=1, N=n_assets, ld=(n_assets + 15) // 16 * 16, D=mkt.n_days, Rw=0, n_mcm=2, R=R,
                        hf_extra_rows=R // 8 + 64, has_caps=1, has_mcm_w=0, ws_limit=24 << 30, reuse_min_windows=32,
                        presum_min_days=8, stride=1)
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
