"""Conjugate prior with missing intraday bars on the GPU: the return rows next to a NaN bar are dropped as the
reference's dropna does (portfolio_calculations.py:314-318), on every route of the batched engine, against the
oracle with the dropna prior of tests/_dropna_ref.py."""
import dataclasses

import numpy as np
import pandas as pd
import pytest

from oracle import bayes_oracle as bo
from tests._dropna_ref import keep_mask, use_dropna_oracle
from tests._golden import relerr

pytestmark = pytest.mark.gpu
TOL = 1e-9
ROUTE_TOL = 1e-11
M = 6                      # BP_SCAL_M
OUTS = ("weights", "S0", "rhs", "scalars", "status")


@pytest.fixture(scope="module")
def engine():
    from incorporating_different_sources_b200.engine import BayesEngine
    eng = BayesEngine(0)
    yield eng
    eng.close()


@pytest.fixture(autouse=True)
def dropna_oracle(monkeypatch):
    use_dropna_oracle(monkeypatch)


def _spec(n, rolling_window=60, freq="daily", strategy="conjugate_hf_vix_vw"):
    return dict(weighting_strategy=strategy, size=n, risk_aversion=5, turnover_cost=15, rebalancing_frequency="daily",
                rolling_window=rolling_window, rolling_window_frequency=freq, mcm_scaling=1, display_name="x")


def _holed(mkt, cells):
    H = mkt.hf_prices.copy()
    for r, c in cells:
        H[r, c] = np.nan
    return dataclasses.replace(mkt, hf_prices=H)


def _holes(mkt, batch, rng, bars, n_iso=40):
    """Holes in first-of-day bars, at hf_lo and hf_hi - 1 of some windows, a whole missing day of one stock and
    isolated bars, all inside the rows the batch reads."""
    N = mkt.n_assets
    lo_all, hi_all = int(batch.hf_lo.min()), int(batch.hf_hi.max())
    day0 = -(-lo_all // bars)
    cells = [(d * bars, int(rng.integers(N))) for d in range(day0, hi_all // bars, 3)]
    for i in range(0, batch.n_windows, 5):
        cells += [(int(batch.hf_lo[i]), int(rng.integers(N))), (int(batch.hf_hi[i]) - 1, int(rng.integers(N)))]
    whole = day0 + 2
    cells += [(r, 1) for r in range(whole * bars, (whole + 1) * bars)]
    cells += [(int(r), int(c)) for r, c in zip(rng.integers(lo_all, hi_all, n_iso), rng.integers(0, N, n_iso))]
    return _holed(mkt, cells)


def _check_oracle(got, spec, mkt, d_idx, check, look, tol=TOL):
    cols = np.arange(mkt.n_assets)
    keep = keep_mask(mkt.hf_prices)
    for i in check:
        ref = bo.conjugate_window(spec, mkt, d_idx[i], cols, hf_lookback_days=look)
        lo, hi = bo.hf_window_rows(spec, mkt.hf_ts, mkt.dates[d_idx[i]], look)
        assert ref["hf_returns"] == keep[lo + 1:hi].sum()
        s = got["scalars"][i]
        assert got["status"][i] == 0, i
        assert s[M] == ref["hf_returns"], i
        assert relerr(got["weights"][i], ref["weights"]) <= tol, i
        if "S0" in got:
            assert relerr(got["S0"][i], ref["S0"]) <= tol, i
        if "rhs" in got:
            assert relerr(got["rhs"][i], ref["c"] * (ref["S0"] @ ref["w0"]) + ref["t"]) <= tol, i
        assert abs(s[0] - ref["n0"]) <= tol * ref["n0"]
        assert abs(s[4] - ref["c"]) <= tol * abs(ref["c"])
        assert abs(s[5] - ref["v0"]) <= tol * abs(ref["v0"])


def _close_routes(a, b):
    assert np.array_equal(a["status"], b["status"])
    assert np.array_equal(a["scalars"][:, M], b["scalars"][:, M])
    for k in ("weights", "S0", "rhs"):
        if k in a and k in b:
            assert relerr(a[k], b[k]) <= ROUTE_TOL, k


def test_parity_one_tile_per_day_with_holes(engine):
    from incorporating_different_sources_b200.engine import upload_synthetic
    from incorporating_different_sources_b200.synthetic import generate_market
    from incorporating_different_sources_b200.windows import plan_daily_windows
    n, W = 24, 40
    base = generate_market(n, 120, seed=101)
    spec = _spec(n)
    d_idx = list(range(120 - W, 120))
    batch = plan_daily_windows(spec, base.dates, d_idx, base.hf_ts, hf_lookback_days=7)
    mkt = _holes(base, batch, np.random.default_rng(1), 78)
    upload_synthetic(engine, mkt)
    got = engine.conjugate(batch, outputs=OUTS)
    assert (got["scalars"][:, M] < batch.hf_hi - batch.hf_lo - 1).all()       # every window lost rows
    _check_oracle(got, spec, mkt, d_idx, range(W), 7)
    # reuse off: every window contracts its own rows
    try:
        engine.set_reuse_min_windows(2 ** 31 - 1)
        alone = engine.conjugate(batch, outputs=OUTS)
    finally:
        engine.set_reuse_min_windows(32)
    _close_routes(alone, got)
    _check_oracle(alone, spec, mkt, d_idx, range(0, W, 7), 7)


def test_presummed_day_blocks_with_holes(engine):
    from incorporating_different_sources_b200.engine import upload_synthetic
    from incorporating_different_sources_b200.synthetic import generate_market
    from incorporating_different_sources_b200.windows import plan_daily_windows
    n, W, look = 40, 24, 366
    base = generate_market(n, 270 + W, seed=102)
    spec = _spec(n, rolling_window=252)
    d_idx = list(range(270, 270 + W))
    batch = plan_daily_windows(spec, base.dates, d_idx, base.hf_ts, hf_lookback_days=look)
    mkt = _holes(base, batch, np.random.default_rng(2), 78, n_iso=400)
    upload_synthetic(engine, mkt)
    outs = ("weights", "rhs", "scalars", "status")
    try:
        engine.set_hf_presum_min_days(0)
        plain = engine.conjugate(batch, outputs=outs)
        engine.set_hf_presum_min_days(8)
        got = engine.conjugate(batch, outputs=outs)
    finally:
        engine.set_hf_presum_min_days(8)
    _close_routes(got, plain)
    _check_oracle(got, spec, mkt, d_idx, range(0, W, 6), look)
    n0, S0 = engine.hf_cov(plan_daily_windows(spec, base.dates, d_idx[:3], base.hf_ts, hf_lookback_days=look))
    for i in range(3):
        assert relerr(S0[i], bo.conjugate_window(spec, mkt, d_idx[i], np.arange(n), hf_lookback_days=look)["S0"]) <= TOL


@pytest.mark.parametrize("look", [7, 31])
def test_irregular_calendar_with_holes(engine, look):
    from incorporating_different_sources_b200.synthetic import generate_market
    from incorporating_different_sources_b200.windows import ffill_rows, plan_daily_windows
    n, W, nwin, B = 24, 40, 60, 26
    base = generate_market(n, 40 + nwin + W, seed=103, bars_per_day=B)
    rng = np.random.default_rng(6)
    keep = np.ones(len(base.hf_ts), dtype=bool)
    for day in rng.choice(base.n_days, size=12, replace=False):
        keep[day * B + 13:(day + 1) * B] = False               # half days
    keep[rng.choice(len(keep), size=60, replace=False)] = False  # bars absent from the calendar
    base = dataclasses.replace(base, hf_ts=base.hf_ts[keep], hf_prices=np.ascontiguousarray(base.hf_prices[keep]))
    spec = _spec(n, rolling_window=nwin, strategy="conjugate_hf_epu_vw")
    d_idx = list(range(base.n_days - W, base.n_days))
    batch = plan_daily_windows(spec, base.dates, d_idx, base.hf_ts, hf_lookback_days=look)
    lo, hi = int(batch.hf_lo.min()), int(batch.hf_hi.max())
    cells = [(int(r), int(c)) for r, c in zip(rng.integers(lo, hi, 80), rng.integers(0, n, 80))]
    cells += [(int(r), 2) for r in batch.hf_lo[::4]] + [(int(r) - 1, 3) for r in batch.hf_hi[::4]]
    mkt = _holed(base, cells)
    engine.upload_market(prices=mkt.prices, rf_row=ffill_rows(mkt.dates, mkt.dates, mkt.rf), caps=mkt.caps,
                         hf_prices=mkt.hf_prices, mcm=np.stack([mkt.vix, mkt.epu]))
    got = engine.conjugate(batch, outputs=OUTS)
    _check_oracle(got, spec, mkt, d_idx, range(W), look)


@pytest.mark.parametrize("n", [200, 520])
def test_streaming_prep_narrow_and_wide_with_holes(engine, n):
    """N <= 512: one pass over the intraday rows; N > 512: two column passes that centre y in place."""
    from incorporating_different_sources_b200.engine import upload_synthetic
    from incorporating_different_sources_b200.synthetic import generate_market
    from incorporating_different_sources_b200.windows import plan_daily_windows
    W = 4
    base = generate_market(n, 300, seed=104)
    spec = _spec(n, rolling_window=252)
    d_idx = list(range(300 - 3 * W, 300, 3))        # sparse dates: no block reuse, every window streams its rows
    batch = plan_daily_windows(spec, base.dates, d_idx, base.hf_ts, hf_lookback_days=7)
    mkt = _holes(base, batch, np.random.default_rng(3), 78)
    upload_synthetic(engine, mkt)
    got = engine.conjugate(batch, outputs=("weights", "rhs", "scalars", "status"))
    _check_oracle(got, spec, mkt, d_idx, range(W), 7)


def test_weekly_windows_with_holes(engine):
    from incorporating_different_sources_b200.engine import upload_synthetic
    from incorporating_different_sources_b200.synthetic import generate_market
    from incorporating_different_sources_b200.windows import plan_weekly_windows
    n, W = 20, 30
    base = generate_market(n, 460, seed=105)
    spec = _spec(n, rolling_window=70, freq="weekly", strategy="conjugate_hf_epu_vw")
    d_idx = list(range(460 - W, 460))
    rows, cb = plan_weekly_windows(spec, base.dates, d_idx, base.dates, base.rf, np.stack([base.vix, base.epu]), base.hf_ts)
    mkt = _holes(base, cb, np.random.default_rng(4), 78)
    upload_synthetic(engine, mkt)
    engine.set_resampled(rows)
    got = engine.conjugate(cb, outputs=("weights", "scalars", "status"))
    _check_oracle(got, spec, mkt, d_idx, range(W), None)


def test_pipelined_upload_with_holes_at_segment_boundaries(engine):
    """Holes on both sides of every segment boundary of a segmented asynchronous upload: return row b, the first of a
    segment, reads price row b - 1 of the previous one.  The pipelined call and sub-batches cut along the segments
    (which wait for their own segments only) are bit-identical to the blocking upload."""
    import torch
    from incorporating_different_sources_b200.synthetic import generate_market
    from incorporating_different_sources_b200.windows import ffill_rows, plan_daily_windows, split_batch_by_fractions
    n, n_days, segs = 40, 200, 4
    base = generate_market(n, n_days, seed=106)
    spec = _spec(n)
    d_idx = list(range(60, n_days))
    R = base.hf_prices.shape[0]
    bounds = [R - (R >> (s + 1)) for s in range(segs - 1)]      # the library's geometric segments
    cells = []
    for k, b in enumerate(bounds):
        cells += [(b - 1, k), (b, k + 5), (b - 2, k + 10), (b + 1, k + 15)]
    mkt = _holed(base, cells)
    keep = keep_mask(mkt.hf_prices)
    assert not keep[np.array(bounds)].any() and not keep[np.array(bounds) + 1].any()
    arrays = dict(prices=mkt.prices, caps=mkt.caps, hf_prices=mkt.hf_prices, mcm=np.stack([mkt.vix, mkt.epu]),
                  rf_row=ffill_rows(mkt.dates, mkt.dates, mkt.rf))
    batch = plan_daily_windows(spec, mkt.dates, d_idx, mkt.hf_ts, hf_lookback_days=7)
    outs = ("weights", "scalars", "status", "w1")
    engine.upload_market(**arrays)
    ref = engine.conjugate(batch, outputs=outs)
    fr = [1 - 0.5 ** (s + 1) for s in range(segs - 1)]
    parts = split_batch_by_fractions(batch, fr, R)
    assert len(parts) > 2
    ref_parts = [engine.conjugate(sub, outputs=("weights", "S0", "scalars")) for _, _, sub in parts]
    hit = [i for i in range(batch.n_windows) if any(batch.hf_lo[i] < b < batch.hf_hi[i] for b in bounds)]
    assert hit
    _check_oracle(ref, spec, mkt, d_idx, hit[::3], 7)
    pinned = {k: torch.from_numpy(np.ascontiguousarray(v)).pin_memory() for k, v in arrays.items()}
    try:
        engine.set_upload_pipeline(segs, 0)
        engine.upload_market(**{k: v.numpy() for k, v in pinned.items()}, async_copy=True)
        got = engine.conjugate(batch, outputs=outs)
        engine.synchronize()
        for k in outs:
            assert np.array_equal(got[k], ref[k]), k
        engine.upload_market(**{k: v.numpy() for k, v in pinned.items()}, async_copy=True)
        for (_, _, sub), want in zip(parts, ref_parts):
            g = engine.conjugate(sub, outputs=("weights", "S0", "scalars"))       # S0: not the pipelined path
            for k in want:
                assert np.array_equal(g[k], want[k]), k
        engine.synchronize()
    finally:
        engine.set_upload_pipeline()


def test_nan_outside_the_windows_changes_nothing(engine):
    """NaN bars in pool columns that are not selected, or in intraday rows no window reads, drop nothing: the result
    is bit-identical to the clean market."""
    from incorporating_different_sources_b200.engine import upload_synthetic
    from incorporating_different_sources_b200.synthetic import generate_market
    from incorporating_different_sources_b200.windows import ffill_rows, plan_daily_windows
    n_pool, n = 32, 16
    mkt = generate_market(n_pool, 120, seed=107)
    spec = _spec(n)
    d_idx = list(range(90, 120))
    cols = np.arange(0, 2 * n, 2)
    rf_row = ffill_rows(mkt.dates, mkt.dates, mkt.rf)
    prior_n = np.full(len(d_idx), 150.0)

    def run_pool(H):
        engine.upload_pool(prices=mkt.prices, rf_row=rf_row, caps=mkt.caps, hf_prices=H)
        engine.select_market(cols, 0, mkt.n_days, 0, H.shape[0])
        b = plan_daily_windows(spec, mkt.dates, d_idx, mkt.hf_ts, hf_lookback_days=7)
        b.prior_n = prior_n
        out = engine.conjugate(b, outputs=OUTS)
        engine.upload_pool(None, None)
        return out

    clean = run_pool(mkt.hf_prices)
    H = mkt.hf_prices.copy()
    H[::7, 1::2] = np.nan                                   # every odd (unselected) column is full of holes
    dirty = run_pool(H)
    for k in OUTS:
        assert np.array_equal(dirty[k], clean[k]), k

    sub = _spec(n_pool)
    batch = plan_daily_windows(sub, mkt.dates, d_idx, mkt.hf_ts, hf_lookback_days=7)
    upload_synthetic(engine, mkt)
    clean = engine.conjugate(batch, outputs=OUTS)
    lo, hi = int(batch.hf_lo.min()), int(batch.hf_hi.max())
    H = mkt.hf_prices.copy()
    H[:lo:3, :] = np.nan                                    # price rows before the first window's first bar
    H[hi::5, 4] = np.nan                                    # and after the last window's last bar
    upload_synthetic(engine, dataclasses.replace(mkt, hf_prices=H))
    dirty = engine.conjugate(batch, outputs=OUTS)
    for k in OUTS:
        assert np.array_equal(dirty[k], clean[k]), k


def test_windows_with_fewer_than_two_returns(engine):
    """A window left with m = 0 or 1 returns: NaN S0 and weights, BP_SCAL_M = m, a non-zero status, and the other
    windows bit-identical to the batch without it (one-day look-backs do not share bars)."""
    from incorporating_different_sources_b200.engine import upload_synthetic
    from incorporating_different_sources_b200.synthetic import generate_market
    from incorporating_different_sources_b200.windows import plan_daily_windows, slice_batch
    n = 10
    base = generate_market(n, 120, seed=108)
    spec = _spec(n)
    d_idx = list(range(80, 120, 2))
    batch = plan_daily_windows(spec, base.dates, d_idx, base.hf_ts, hf_lookback_days=1)
    H = base.hf_prices.copy()
    bad = {3: 0, 11: 1}
    lo, hi = int(batch.hf_lo[3]), int(batch.hf_hi[3])
    H[lo:hi:2, 0] = np.nan                                  # every return of window 3 touches a hole
    lo, hi = int(batch.hf_lo[11]), int(batch.hf_hi[11])
    H[lo:hi - 2, 5] = np.nan                                # window 11 keeps its last return only
    H[int(batch.hf_lo[7]) + 9, 2] = np.nan                  # a neighbour with an ordinary hole
    mkt = dataclasses.replace(base, hf_prices=H)
    upload_synthetic(engine, mkt)
    try:
        engine.set_reuse_min_windows(2 ** 31 - 1)
        got = engine.conjugate(batch, outputs=OUTS)
        good = [i for i in range(batch.n_windows) if i not in bad]
        parts = [slice_batch(batch, 0, 3), slice_batch(batch, 4, 11), slice_batch(batch, 12, batch.n_windows)]
        rest = [engine.conjugate(p, outputs=OUTS) for p in parts]
    finally:
        engine.set_reuse_min_windows(32)
    for i, m in bad.items():
        assert got["scalars"][i][M] == m
        assert got["status"][i] != 0
        assert np.isnan(got["S0"][i]).all() and np.isnan(got["weights"][i]).all()
    for k in OUTS:
        assert np.array_equal(np.concatenate([r[k] for r in rest]), got[k][good]), k
    _check_oracle({k: got[k][good] for k in OUTS}, spec, mkt, [d_idx[i] for i in good], range(len(good)), 1)


def _frames(md, names, d):
    caps_df = md["stock_market_caps_df"][names].loc[:d]
    prices_df = md["stock_prices_df"][names].loc[:d]
    intr_df = md["stock_intraday_prices_df"][names]
    intr_df = intr_df.loc[intr_df.index <= d.replace(hour=23, minute=59, second=59)]
    return caps_df, prices_df, intr_df


def test_facade_with_missing_bars():
    from incorporating_different_sources_b200 import portfolio_calculations as pc
    from incorporating_different_sources_b200.synthetic import generate_market
    n = 10
    base = generate_market(n, 300, seed=109)
    spec = _spec(n, rolling_window=252)
    cols = np.arange(n)
    checks = []
    for d_idx in (280, 290):
        lo, hi = bo.hf_window_rows(spec, base.hf_ts, base.dates[d_idx])
        checks.append((d_idx, [(lo, 1), (lo + 1, 2), (lo + 30, 4), (lo + 31, 4), (hi - 1, 7)]))
    mkt = _holed(base, [c for _, cs in checks for c in cs])
    md = mkt.market_data()
    names = list(md["stock_prices_df"].columns)
    for d_idx, _ in checks:
        d = pd.Timestamp(mkt.dates[d_idx])
        caps_df, prices_df, intr_df = _frames(md, names, d)
        vix = md["vix_prices_df"].loc[md["vix_prices_df"].index <= d]
        ref = bo.conjugate_window(spec, mkt, d_idx, cols)
        S0 = pc.calculate_conjugate_prior_S(spec, d, intr_df, vix)
        assert relerr(S0.loc[names, names].to_numpy(), ref["S0"]) <= TOL
        w = pc.calculate_conjugate_hf_mcm_portfolio(spec, d, caps_df, prices_df, intr_df, vix, md["risk_free_rate_df"])
        assert list(w.index) == names and relerr(w["Weight"].to_numpy(), ref["weights"]) <= TOL
    # m < 2: the prior is all NaN (pandas' cov) and the posterior raises the reference's ValueError (:492-494)
    d_idx = 295
    lo, hi = bo.hf_window_rows(spec, base.hf_ts, base.dates[d_idx])
    H = base.hf_prices.copy()
    H[lo:hi - 2, 3] = np.nan
    md = dataclasses.replace(base, hf_prices=H).market_data()
    d = pd.Timestamp(base.dates[d_idx])
    caps_df, prices_df, intr_df = _frames(md, names, d)
    vix = md["vix_prices_df"].loc[md["vix_prices_df"].index <= d]
    assert np.isnan(pc.calculate_conjugate_prior_S(spec, d, intr_df, vix).to_numpy()).all()
    with pytest.raises(ValueError, match="conjugate_posterior_w_df contains NaN values"):
        pc.calculate_conjugate_hf_mcm_portfolio(spec, d, caps_df, prices_df, intr_df, vix, md["risk_free_rate_df"])
    with pytest.raises(ValueError, match="conjugate_posterior_w_df contains NaN values"):
        pc.calculate_conjugate_posterior_w(spec, d, prices_df, caps_df, intr_df, vix, md["risk_free_rate_df"])


@pytest.mark.parametrize("freq", ["daily", "weekly"])
def test_backtest_with_missing_bars(engine, freq):
    """The loop level no longer refuses held stocks with missing bars; its per-date weights match the oracle."""
    from incorporating_different_sources_b200 import backtest as bt
    from incorporating_different_sources_b200 import portfolio_calculations as pc
    from incorporating_different_sources_b200.synthetic import generate_market
    n = 8
    base = generate_market(n, 330, seed=110)
    rng = np.random.default_rng(9)
    R = base.hf_prices.shape[0]
    first = 200 * 78
    cells = [(int(r), int(c)) for r, c in zip(rng.integers(first, R, 300), rng.integers(0, n, 300))]
    cells += [(r, 6) for r in range(300 * 78, 301 * 78)]          # one stock misses a whole day
    mkt = _holed(base, cells)
    md = mkt.market_data()
    spec = dict(_spec(n, rolling_window=150 if freq == "daily" else 40, freq=freq), rebalancing_frequency="weekly")
    look = 7
    start, end = pd.Timestamp(mkt.dates[260]), pd.Timestamp(mkt.dates[-1])
    res = pc.backtest_portfolio(spec, start, end, md, engine=engine, hf_lookback_days=look)
    assert np.isfinite(res["portfolio_simple_returns_series"].to_numpy()).all()
    dates_all = md["stock_prices_df"].index
    in_range = np.nonzero((dates_all >= start) & (dates_all <= end))[0]
    reb_pos = list(in_range[bt.rebalance_flags(dates_all[in_range], spec["rebalancing_frequency"])])
    universes, _, _ = bt.select_universes(md["stock_market_caps_df"], md["stock_prices_df"], md["stock_intraday_prices_df"],
                                          dates_all[reb_pos], n, bt.get_window_trading_days(spec), spec["rebalancing_frequency"])
    W, _ = bt._batched_weights(engine, spec, md, dates_all, reb_pos, universes, look)
    engine.upload_pool(None, None)
    keep = keep_mask(mkt.hf_prices)
    dropped = 0
    for r, d_idx in enumerate(reb_pos):
        cols = np.array(sorted(names_to_pos(md, universes[r])))
        ref, _ = bo.window_weights(spec, mkt, d_idx, cols, hf_lookback_days=look)
        assert relerr(W[r, cols], ref) <= TOL, r
        lo, hi = bo.hf_window_rows(spec, mkt.hf_ts, mkt.dates[d_idx], look)
        dropped += (~keep[lo + 1:hi]).sum()
    assert dropped > 0


def names_to_pos(md, names):
    pos = {c: i for i, c in enumerate(md["stock_prices_df"].columns)}
    return [pos[s] for s in names]
