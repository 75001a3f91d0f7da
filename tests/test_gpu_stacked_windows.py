"""Stacked working markets on the GPU: windows with different asset sets in one batched call (``select_windows``)
give the same bits as one ``select_market`` slice and one call per window, on every strategy of the loop level,
daily and weekly; the routes that share work between windows stay off; backtests give the same bits with stacking
on and off."""
import ctypes as C
import itertools
import json
import os

import numpy as np
import pandas as pd
import pytest

from oracle import bayes_oracle as bo
from tests._golden import relerr

pytestmark = pytest.mark.gpu
TOL = 1e-9
GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
POOL, DAYS = 160, 760
STRATS = ["vw", "ew", "conjugate_hf_vix_vw", "conjugate_hf_epu_ew", "jeffreys", "jorion", "shrinkage"]
SOLVE_OUTS = ("weights", "nu", "w1", "scalars", "status")


@pytest.fixture(scope="module")
def engine():
    from incorporating_different_sources_b200.engine import BayesEngine
    eng = BayesEngine(0)
    yield eng
    eng.close()


@pytest.fixture(scope="module")
def mkt():
    from incorporating_different_sources_b200.synthetic import generate_market
    return generate_market(POOL, DAYS, seed=41)


def _upload(engine, mkt, H=None):
    from incorporating_different_sources_b200.windows import ffill_rows
    engine.upload_pool(prices=mkt.prices, rf_row=ffill_rows(mkt.dates, mkt.dates, mkt.rf), caps=mkt.caps,
                       hf_prices=mkt.hf_prices if H is None else H)


def _spec(strat, N, freq):
    if strat in ("vw", "ew"):        # what the backtest evaluates for vw / ew: the prior weights w0 of a 3-price window
        return dict(weighting_strategy="conjugate_hf_vix_" + strat, size=N, mcm_scaling=1, rolling_window=3,
                    rolling_window_frequency="daily", risk_aversion=1)
    return dict(weighting_strategy=strat, size=N, mcm_scaling=1, risk_aversion=5,
                rolling_window=150 if freq == "daily" else 140, rolling_window_frequency=freq)


def _plan(spec, mkt, d_idx, look, **offsets):
    from incorporating_different_sources_b200.windows import plan_daily_windows, plan_weekly_windows
    need_hf = spec["weighting_strategy"].startswith("conjugate")
    if spec["rolling_window_frequency"] == "weekly":
        return plan_weekly_windows(spec, mkt.dates, d_idx, mkt.dates, mkt.rf, None, mkt.hf_ts if need_hf else None,
                                   hf_lookback_days=look, need_hf=need_hf)
    return None, plan_daily_windows(spec, mkt.dates, d_idx, mkt.hf_ts if need_hf else None, hf_lookback_days=look,
                                    need_hf=need_hf, **offsets)


def _call(engine, strat, batch, prior_n):
    if strat in ("vw", "ew"):
        batch.prior_n = prior_n
        return engine.moments(batch, outputs=("w0", "t", "scalars"))
    if strat.startswith("conjugate"):
        batch.prior_n = prior_n
        return engine.conjugate(batch, outputs=SOLVE_OUTS)
    return {"jeffreys": engine.jeffreys, "jorion": engine.jorion, "shrinkage": engine.shrinkage}[strat](batch, outputs=SOLVE_OUTS)


def _stacked(engine, strat, spec, mkt, d_idx, cols, look, prior_n):
    from incorporating_different_sources_b200.windows import stack_windows
    rows, plan = _plan(spec, mkt, d_idx, look)
    stk = stack_windows(plan, rows)
    hf = None if stk.hf_lo is None else np.stack([stk.hf_lo, stk.hf_hi], axis=1)
    engine.select_windows(cols, np.stack([stk.day_lo, stk.day_hi], axis=1), hf)
    if stk.resampled is not None:
        engine.set_resampled(stk.resampled)
    return _call(engine, strat, stk.batch, prior_n)


def _per_window(engine, strat, spec, mkt, d_idx, cols, look, prior_n):
    """One select_market slice and one batched call per window, as the backtest's per-set route makes them."""
    out = []
    n = spec["rolling_window"]
    need_hf = spec["weighting_strategy"].startswith("conjugate")
    for i, d in enumerate(d_idx):
        if spec["rolling_window_frequency"] == "weekly":
            engine.select_market(cols[i], 0, mkt.n_days, 0, mkt.hf_prices.shape[0] if need_hf else 0)
            rows, b = _plan(spec, mkt, [d], look)
            engine.set_resampled(rows)
        else:
            _, full = _plan(spec, mkt, [d], look)
            hf_lo = max(int(full.hf_lo[0]) - 1, 0) if need_hf else 0
            hf_hi = int(full.hf_hi[0]) if need_hf else 0
            engine.select_market(cols[i], d - (n - 1), d + 1, hf_lo, hf_hi)
            _, b = _plan(spec, mkt, [d], look, row_offset=d - (n - 1), hf_row_offset=hf_lo)
        out.append(_call(engine, strat, b, prior_n[i:i + 1]))
    return {k: np.concatenate([o[k] for o in out]) for k in out[0]}


def _windows(rng, N, freq, W=6):
    lo = 720 if freq == "weekly" else 160
    d_idx = sorted(int(d) for d in rng.choice(np.arange(lo, DAYS), W, replace=False))
    cols = np.stack([np.sort(rng.choice(POOL, N, replace=False)) for _ in range(W)]).astype(np.int32)
    return d_idx, cols


def _same(a, b):
    for k in a:
        assert np.array_equal(a[k], b[k], equal_nan=a[k].dtype.kind == "f"), k


@pytest.mark.parametrize("N", [10, 50, 100, 130])
@pytest.mark.parametrize("strat,freq", [(s, f) for s in STRATS for f in ("daily", "weekly")
                                        if f == "daily" or s not in ("vw", "ew")])     # vw / ew windows are daily
def test_stacked_batch_is_bit_identical_to_per_window_calls(engine, mkt, strat, freq, N):
    rng = np.random.default_rng(N * 7 + len(strat) + (freq == "weekly"))
    spec = _spec(strat, N, freq)
    d_idx, cols = _windows(rng, N, freq)
    look = 7 if strat.startswith("conjugate") else None
    prior_n = rng.uniform(100.0, 400.0, len(d_idx))
    # the first two windows against the oracle (the conjugate ones with the oracle's own n0 injected)
    refs = []
    for i in range(2):
        if strat.startswith("conjugate"):
            ref = bo.conjugate_window(spec, mkt, d_idx[i], cols[i], look)
            prior_n[i] = ref["n0"]
            refs.append(ref["weights"])
        elif strat in ("vw", "ew"):
            refs.append(bo.prior_w(spec, mkt.caps[d_idx[i], cols[i]]))
        elif strat == "shrinkage":
            refs.append(bo.shrinkage_window(spec, mkt, d_idx[i], cols[i])["weights"])
        else:
            refs.append(bo.window_weights(spec, mkt, d_idx[i], cols[i])[0])
    _upload(engine, mkt)
    try:
        got = _stacked(engine, strat, spec, mkt, d_idx, cols, look, prior_n)
        want = _per_window(engine, strat, spec, mkt, d_idx, cols, look, prior_n)
    finally:
        engine.upload_pool(None, None)
    _same(got, want)
    key = "w0" if strat in ("vw", "ew") else "weights"
    for i, ref in enumerate(refs):
        assert relerr(got[key][i], ref) <= TOL, i
    if key == "weights":
        assert not got["status"].any()


@pytest.mark.parametrize("strat", ["conjugate_hf_vix_vw", "jeffreys"])
def test_no_route_shares_work_between_stacked_windows(engine, mkt, strat):
    """40 consecutive trade dates: on one working market they take block reuse (conjugate) or the chain (Jeffreys);
    stacked, with one column set per window, every window contracts and factorises its own rows, with the same bits as
    one call per window."""
    rng = np.random.default_rng(5)
    N = 24
    spec = _spec(strat, N, "daily")
    d_idx = list(range(700, 740))
    look = 7 if strat.startswith("conjugate") else None
    prior_n = rng.uniform(100.0, 400.0, len(d_idx))
    _upload(engine, mkt)
    try:
        one = np.arange(N, dtype=np.int32)
        engine.select_market(one, 0, mkt.n_days, 0, mkt.hf_prices.shape[0])
        _, b = _plan(spec, mkt, d_idx, look)
        engine.gram_work(), engine.solve_work()
        _call(engine, strat, b, prior_n)
        shared_gram, shared_solve = engine.gram_work(), engine.solve_work()
        assert shared_gram["add_blocks"] > 0 if strat.startswith("conjugate") else shared_solve["chained"] > 0
        cols = np.stack([np.sort(rng.choice(POOL, N, replace=False)) for _ in d_idx]).astype(np.int32)
        got = _stacked(engine, strat, spec, mkt, d_idx, cols, look, prior_n)
        gram, solve = engine.gram_work(), engine.solve_work()
        assert gram["add_blocks"] == 0 and gram["precompute_rows"] == 0
        assert solve["chained"] == 0 and solve["factored"] == len(d_idx)
        want = _per_window(engine, strat, spec, mkt, d_idx, cols, look, prior_n)
    finally:
        engine.upload_pool(None, None)
    _same(got, want)


def test_nan_bars_drop_rows_of_their_own_window_only(engine, mkt):
    rng = np.random.default_rng(8)
    N, strat = 20, "conjugate_hf_vix_vw"
    spec = _spec(strat, N, "daily")
    d_idx = [600, 600, 650, 651]                 # two windows on the same date read the same pool rows
    cols = np.stack([np.sort(rng.choice(POOL, N, replace=False)) for _ in d_idx]).astype(np.int32)
    only0 = int(np.setdiff1d(cols[0], cols[1])[0])
    _, full = _plan(spec, mkt, d_idx, 7)
    H = mkt.hf_prices.copy()
    lo, hi = int(full.hf_lo[0]), int(full.hf_hi[0])
    H[lo + 5, only0] = np.nan                    # window 0's column, inside the rows windows 0 and 1 both read
    H[lo + 40: lo + 43, only0] = np.nan
    for w in (2, 3):
        H[int(full.hf_lo[w]) + 17, cols[w][3]] = np.nan
    prior_n = rng.uniform(100.0, 400.0, len(d_idx))
    _upload(engine, mkt, H)
    try:
        got = _stacked(engine, strat, spec, mkt, d_idx, cols, 7, prior_n)
        want = _per_window(engine, strat, spec, mkt, d_idx, cols, 7, prior_n)
    finally:
        engine.upload_pool(None, None)
    _same(got, want)
    m = got["scalars"][:, 6]
    span = (full.hf_hi - full.hf_lo - 1).astype(float)
    assert m[0] < span[0] and m[1] == span[1]
    assert m[2] < span[2] and m[3] < span[3]


@pytest.mark.parametrize("strat", ["conjugate_hf_epu_ew", "jeffreys", "jorion"])
@pytest.mark.parametrize("freq", ["daily", "weekly"])
def test_condition_estimate_is_bit_identical(engine, mkt, strat, freq):
    rng = np.random.default_rng(9)
    spec = _spec(strat, 50, freq)
    d_idx, cols = _windows(rng, 50, freq, W=5)
    look = 7 if strat.startswith("conjugate") else None
    prior_n = rng.uniform(100.0, 400.0, len(d_idx))
    _upload(engine, mkt)
    engine.set_condition_estimate(True)
    try:
        got = _stacked(engine, strat, spec, mkt, d_idx, cols, look, prior_n)
        want = _per_window(engine, strat, spec, mkt, d_idx, cols, look, prior_n)
    finally:
        engine.set_condition_estimate(False)
        engine.upload_pool(None, None)
    _same(got, want)
    assert np.all(got["scalars"][:, 11] > 0)


def test_error_paths(engine, mkt):
    from incorporating_different_sources_b200 import _lib
    from incorporating_different_sources_b200.windows import plan_daily_windows
    _upload(engine, mkt)
    R = mkt.hf_prices.shape[0]
    try:
        cols = np.array([[0, 1, 2], [3, 4, 5]], dtype=np.int32)
        with pytest.raises(ValueError, match="column 999 outside"):
            engine.select_windows(np.array([[0, 1, 999], [3, 4, 5]]), [[0, 10], [5, 15]])
        with pytest.raises(ValueError, match="daily row range"):
            engine.select_windows(cols, [[0, 10], [DAYS - 5, DAYS + 1]])
        with pytest.raises(ValueError, match="intraday row range"):
            engine.select_windows(cols, [[0, 10], [5, 15]], [[0, 100], [R - 10, R + 1]])
        # offsets that do not tile the stack (the engine computes them; a direct caller may not)
        lib = _lib.load()
        lo, hi, off = (np.array(a, dtype=np.int32) for a in ([0, 5], [10, 15], [0, 11]))
        sel = _lib.WindowSelect()
        sel.n_windows, sel.n_cols = 2, 3
        sel.cols, sel.day_lo, sel.day_hi, sel.day_off = cols.ctypes.data, lo.ctypes.data, hi.ctypes.data, off.ctypes.data
        sel.hf_lo = sel.hf_hi = sel.hf_off = None
        assert lib.bp_select_windows(engine._h, C.byref(sel)) == _lib.BP_ERR_INVALID
        assert "tile the stack" in _lib.last_error()
        # a batch that names rows outside the stack
        spec = _spec("jeffreys", 3, "daily")
        spec["rolling_window"] = 5
        engine.select_windows(cols, [[100, 105], [200, 205]])
        b = plan_daily_windows(spec, mkt.dates, [104, 204], need_hf=False)
        b.day_row = np.array([4, 12], dtype=np.int32)
        with pytest.raises(ValueError, match="day_row 12"):
            engine.jeffreys(b)
        b.day_row = np.array([4, 7], dtype=np.int32)             # inside the stack, but across two windows' blocks
        with pytest.raises(ValueError, match="window 1 reads stack rows outside one window's block"):
            engine.jeffreys(b)
        b.day_row = np.array([4, 9], dtype=np.int32)
        assert not engine.jeffreys(b)["status"].any()          # the handle is still usable
    finally:
        engine.upload_pool(None, None)


@pytest.mark.parametrize("N", [12289, 25000])
def test_wide_selections_equal_direct_upload(engine, N):
    """Working markets wider than the 12,288 columns the gather stages in shared memory at a time: a select_market slice
    and each window of a select_windows stack give the excess returns (prices and risk-free rate) that a direct upload
    of the same columns gives, bit for bit."""
    from incorporating_different_sources_b200.windows import plan_daily_windows, slice_batch, stack_windows
    rng = np.random.default_rng(N)
    P, D, H, n = N + 1000, 40, 30, 20
    dates = np.busday_offset("2020-01-01", np.arange(D), roll="forward").astype("datetime64[ns]")
    prices = 100.0 * np.exp(np.cumsum(rng.normal(0.0, 0.01, (D, P)), axis=0))
    caps = prices * rng.uniform(1e6, 1e9, P)
    hf = rng.uniform(50.0, 150.0, (H, P))
    rf = rng.uniform(0.0, 1e-4, D)
    spec = dict(weighting_strategy="jeffreys", rolling_window=n, rolling_window_frequency="daily", risk_aversion=1)
    d_idx = [25, 39]
    cols = np.stack([rng.permutation(P)[:N] for _ in d_idx]).astype(np.int32)
    plan = plan_daily_windows(spec, dates, d_idx, need_hf=False)
    want = []
    for w in range(len(d_idx)):
        engine.upload_market(prices=prices[:, cols[w]], rf_row=rf, caps=caps[:, cols[w]], hf_prices=hf[:, cols[w]])
        want.append(engine.excess_returns(slice_batch(plan, w, w + 1)))
    engine.upload_pool(prices=prices, rf_row=rf, caps=caps, hf_prices=hf)
    try:
        for w, d in enumerate(d_idx):
            engine.select_market(cols[w], d - (n - 1), d + 1, 0, H)
            b = plan_daily_windows(spec, dates, [d], need_hf=False, row_offset=d - (n - 1))
            assert np.array_equal(engine.excess_returns(b), want[w]), w
        stk = stack_windows(plan)
        engine.select_windows(cols, np.stack([stk.day_lo, stk.day_hi], axis=1), [[0, H], [5, H]])
        for w in range(len(d_idx)):
            assert np.array_equal(engine.excess_returns(slice_batch(stk.batch, w, w + 1)), want[w]), w
    finally:
        engine.upload_pool(None, None)


# ------------------------------------------------------------------ backtest level: stacking on == stacking off
def _backtest_both(engine, spec, md, start, end, **kw):
    from incorporating_different_sources_b200 import portfolio_calculations as pc
    out = []
    for n in (15, 0):
        engine.set_stack_max_windows(n)
        tm, diag = {}, {}
        try:
            res = pc.backtest_portfolio(spec, start, end, md, engine=engine, timings=tm, diagnostics=diag, **kw)
        finally:
            engine.set_stack_max_windows()
        out.append((res, diag["rcond"], tm))
    (a, ra, ta), (b, rb, tb) = out
    for k in a:
        assert a[k].index.equals(b[k].index), k
        assert np.array_equal(a[k].to_numpy(), b[k].to_numpy(), equal_nan=True), k
    assert ra.index.equals(rb.index) and np.array_equal(ra.to_numpy(), rb.to_numpy(), equal_nan=True)
    assert tb["stacked_windows"] == 0 and tb["stacked_calls"] == 0
    return ta


@pytest.mark.parametrize("strat", ["conjugate_hf_vix_vw", "jeffreys"])
def test_backtest_scaled_down_shipped_spec(engine, strat):
    """Top 6 of 12, monthly rebalancing, weekly windows: nearly every rebalance date has a universe of its own."""
    from incorporating_different_sources_b200.synthetic import generate_market
    mkt = generate_market(12, 520, seed=43)
    spec = dict(weighting_strategy=strat, size=6, risk_aversion=5, turnover_cost=15, rebalancing_frequency="monthly",
                rolling_window=30, rolling_window_frequency="weekly", mcm_scaling=1, display_name="shipped, scaled down")
    tm = _backtest_both(engine, spec, mkt.market_data(), pd.Timestamp(mkt.dates[200]), pd.Timestamp(mkt.dates[-1]))
    assert tm["stacked_windows"] == tm["rebalances"] and tm["stacked_calls"] >= 1


@pytest.mark.parametrize("strat", ["jeffreys", "conjugate_hf_epu_ew", "shrinkage", "jorion", "vw"])
def test_backtest_small_and_large_sets_mix(engine, strat, monkeypatch):
    """Daily top-5 backtest: one universe for the first 40 dates (its own call, with the routes that share work), then
    a universe that changes every date (stacked), with four or five stocks: small sets of two N."""
    from incorporating_different_sources_b200 import backtest as bt
    from incorporating_different_sources_b200.synthetic import generate_market
    mkt = generate_market(9, 260, seed=44)
    md = mkt.market_data()
    start = 150
    # universes without stock 0: 56 of five stocks, and 70 of four, where the top 5 has only 4 stocks (another N)
    combos = list(itertools.combinations(range(1, 9), 5)) + list(itertools.combinations(range(1, 9), 4))

    def provider(d):
        i = int(np.searchsorted(mkt.dates, np.datetime64(d))) - start
        return [mkt.tickers[c] for c in ([0, 1, 2, 3, 4] if i < 40 else combos[(7 * i) % len(combos)])]

    monkeypatch.setattr(bt, "UNIVERSE_PROVIDER", provider)
    spec = dict(weighting_strategy=strat, size=5, risk_aversion=5, turnover_cost=15, rebalancing_frequency="daily",
                rolling_window=60, rolling_window_frequency="daily", mcm_scaling=1, display_name="mix")
    tm = _backtest_both(engine, spec, md, pd.Timestamp(mkt.dates[start]), pd.Timestamp(mkt.dates[-1]), hf_lookback_days=7)
    assert 0 < tm["stacked_windows"] < tm["rebalances"]


def test_backtest_late_listing_market(engine):
    from incorporating_different_sources_b200.synthetic import generate_market
    from tests.golden.make_backtest_golden import apply_damage
    z = np.load(os.path.join(GOLD, "bt_jeffreys_daily_top5of8_late_listing.npz"))
    meta = json.loads(str(z["meta"]))
    md = generate_market(**meta["market"]).market_data()
    if meta.get("damage"):
        md = apply_damage(md, meta["damage"])
    tm = _backtest_both(engine, meta["spec"], md, pd.Timestamp(meta["start"]), pd.Timestamp(meta["end"]))
    assert tm["stacked_windows"] > 0
