"""Host-side index logic against the UNMODIFIED reference, on the edge cases the domain has: late listings (NaN
prices inside the look-back), stocks without intraday data, NaN and TIED market caps, a constituent list that names
unknown tickers, portfolios larger than the eligible universe, partially overlapping turnover frames.

Runs on the CPU (no CUDA call); the tests that import the reference's own functions run where its sources are found
(``$REF_SRC``, see oracle/ref_import.py). Index order and membership are compared exactly.
"""
import numpy as np
import pandas as pd
import pytest

from incorporating_different_sources_b200 import backtest as bt
from incorporating_different_sources_b200.synthetic import generate_market
from oracle.ref_import import load_reference, reference_available, set_universe

needs_reference = pytest.mark.skipif(not reference_available(), reason="reference sources not present on this machine")


def _damaged_market():
    mkt = generate_market(12, 90, seed=4242, bars_per_day=4)
    md = mkt.market_data()
    prices, caps, intr = md["stock_prices_df"].copy(), md["stock_market_caps_df"].copy(), md["stock_intraday_prices_df"].copy()
    t = mkt.tickers
    prices.iloc[:70, 1] = np.nan                      # late listing: NaN inside a 30-day look-back until day 100
    prices.iloc[40, 2] = np.nan                       # one hole in the middle of the history
    intr.iloc[:, 3] = np.nan                          # never traded intraday
    intr.loc[intr.index >= prices.index[80], t[4]] = np.nan    # intraday feed stops before the last dates
    caps.iloc[:, 5] = np.nan                          # no market cap at all
    caps.iloc[:, 6] = caps.iloc[:, 7]                 # exact ties on every date
    caps = caps.drop(columns=[t[8]])                  # not in the cap frame
    return mkt, prices, caps, intr


@needs_reference
@pytest.mark.parametrize("freq", ["daily", "weekly", "monthly"])
@pytest.mark.parametrize("size", [3, 7, 50])
def test_universe_selection_matches_reference(freq, size):
    pc = load_reference(check=True)
    mkt, prices, caps, intr = _damaged_market()
    universe = list(mkt.tickers[:11]) + ["ZZZ_UNKNOWN"]          # ticker 11 is not a constituent, one name is unknown
    set_universe(universe)
    bt.UNIVERSE_PROVIDER = lambda d: universe
    try:
        for pos in (45, 69, 71, 79, 83, 89):
            d = prices.index[pos]
            for window_days in (5, 30):
                ref = pc.get_k_largest_stocks_market_caps(caps, prices, intr, d, size, window_days, freq)
                got = bt.get_k_largest_stocks_market_caps(caps, prices, intr, d, size, window_days, freq)
                assert list(got.index) == list(ref.index), (freq, size, pos, window_days)
                assert np.array_equal(got.to_numpy(), ref.to_numpy())
                assert got.name == ref.name and got.dtype == ref.dtype
    finally:
        bt.UNIVERSE_PROVIDER = None


@needs_reference
@pytest.mark.parametrize("freq", ["daily", "weekly", "monthly"])
@pytest.mark.parametrize("size", [3, 7, 50])
def test_vectorised_universe_selection_matches_reference_on_every_date(freq, size):
    """select_universes (all dates at once: cumulative not-NaN counts, per-day intraday counts, stable argsort) against
    the reference's per-date get_k_largest_stocks_market_caps: membership AND order, every date of the damaged market."""
    pc = load_reference(check=True)
    mkt, prices, caps, intr = _damaged_market()
    universe = list(mkt.tickers[:11]) + ["ZZZ_UNKNOWN"]
    set_universe(universe)
    bt.UNIVERSE_PROVIDER = lambda d: universe
    try:
        dates = prices.index[35:]
        for window_days in (5, 30):
            got, nan_bars, cand = bt.select_universes(caps, prices, intr, dates, size, window_days, freq)
            assert len(got) == len(dates)
            for d, names in zip(dates, got):
                ref = pc.get_k_largest_stocks_market_caps(caps, prices, intr, d, size, window_days, freq)
                assert names == list(ref.index), (freq, size, d, window_days)
            # the feed of ticker 4 stops at day 80: NaN bars inside the look-back from then on, none before
            j = cand.index(mkt.tickers[4])
            assert nan_bars[-1, j] and not nan_bars[0, j]
    finally:
        bt.UNIVERSE_PROVIDER = None


@needs_reference
def test_vectorised_universe_selection_without_provider_and_missing_cap_date():
    pc = load_reference(check=True)
    mkt, prices, caps, intr = _damaged_market()
    set_universe(mkt.tickers)
    dates = prices.index[40:]
    got, _, _ = bt.select_universes(caps, prices, intr, dates, 6, 20, "daily")
    for d, names in zip(dates, got):
        ref = pc.get_k_largest_stocks_market_caps(caps, prices, intr, d, 6, 20, "daily")
        assert names == list(ref.index)
    with pytest.raises(ValueError):
        bt.select_universes(caps.drop(index=dates[3]), prices, intr, dates, 6, 20, "daily")
    with pytest.raises(RuntimeError):
        bt.select_universes(caps, prices, intr, dates, 6, 20, "hourly")


def test_universe_selection_errors_match_reference():
    """The exception types are the reference's; its own function is checked beside ours where its sources are found."""
    mkt, prices, caps, intr = _damaged_market()
    set_universe(mkt.tickers)
    d = prices.index[60]
    fns = [bt.get_k_largest_stocks_market_caps]
    if reference_available():
        fns.insert(0, load_reference(check=True).get_k_largest_stocks_market_caps)
    for fn in fns:
        with pytest.raises(RuntimeError):
            fn(caps, prices, intr, d, 5, 30, "hourly")                              # :637
        with pytest.raises(ValueError):
            fn(caps.drop(index=d), prices, intr, d, 5, 30, "daily")                  # :657


@needs_reference
def test_turnover_and_window_helpers_match_reference():
    pc = load_reference(check=True)
    from incorporating_different_sources_b200 import portfolio_calculations as ours
    rng = np.random.default_rng(3)
    names = [f"S{i}" for i in range(9)]
    for _ in range(20):
        a = rng.choice(names, size=rng.integers(1, 8), replace=False)
        b = rng.choice(names, size=rng.integers(1, 8), replace=False)
        before = pd.DataFrame({"Weight": rng.normal(size=len(a))}, index=pd.Index(a, name="Stock"))
        after = pd.DataFrame({"Weight": rng.normal(size=len(b))}, index=pd.Index(b, name="Stock"))
        ref = pc.compute_portfolio_turnover(before.copy(), after.copy())
        assert bt.compute_portfolio_turnover(before, after) == ref
    for freq in ("daily", "weekly", "monthly"):
        spec = dict(rolling_window=37, rolling_window_frequency=freq)
        assert bt.get_window_trading_days(spec) == pc.get_window_trading_days(spec)                  # :126-134
        assert ours.get_window_annualization_factor(spec) == pc.get_window_annualization_factor(spec)  # :116-124


def test_rebalance_calendar_matches_reference_loop():
    """The rebalance rule lives inside the reference's per-day loop (:1166-1176): replay the loop's own
    bookkeeping on a calendar with holidays and compare the flagged days."""
    days = pd.bdate_range("2010-12-20", periods=140)
    days = days.delete([3, 4, 11, 40, 41, 42, 43, 44, 45, 77])          # holidays, one gap longer than a week
    for freq in ("daily", "weekly", "monthly"):
        last, ref = None, []
        for d in days:                                                   # restated from :1166-1176
            if last is None:
                reb = True
            elif freq == "daily":
                reb = True
            elif freq == "weekly":
                reb = d.weekday() == 2 or (d - last).days > 7
            else:
                reb = d.month != last.month
            ref.append(reb)
            if reb:
                last = d
        assert list(bt.rebalance_flags(days, freq)) == ref
    with pytest.raises(ValueError):
        bt.rebalance_flags(days, "yearly")


@needs_reference
@pytest.mark.parametrize("freq", ["daily", "weekly"])
def test_mcm_prior_n_on_the_series_own_calendar_matches_reference(freq):
    """FRED's daily EPU index has an observation on every CALENDAR day: the reference averages the last n
    observations (daily) / the last n weekly buckets (weekly, Sunday's value) of that calendar (:95-112), not the
    last n trading days.  NaN observations and a missing trade date behave like the reference."""
    from incorporating_different_sources_b200.windows import mcm_prior_n
    pc = load_reference(check=True)
    rng = np.random.default_rng(11)
    cal = pd.date_range("2009-01-01", periods=900, freq="D")
    epu = pd.DataFrame({"EPU": 100.0 * np.exp(0.3 * rng.standard_normal(len(cal)))}, index=cal)
    epu.iloc[[100, 101, 350, 357, 500, 506, 520, 560], 0] = np.nan          # holes inside the windows, Sundays among them
    trade = pd.bdate_range("2010-06-01", periods=120)
    trade = trade[~np.isnan(epu.loc[trade, "EPU"].to_numpy())]
    spec = dict(rolling_window=60 if freq == "daily" else 30, rolling_window_frequency=freq, mcm_scaling=1.7,
                weighting_strategy="conjugate_hf_epu_vw")
    got = mcm_prior_n(spec, epu.index.values, epu["EPU"].to_numpy(), trade.values)
    for i, d in enumerate(trade):
        ref = pc.calculate_conjugate_prior_n(spec, d, epu.loc[epu.index <= d])
        assert abs(got[i] - ref) <= 1e-13 * abs(ref), (freq, d, got[i], ref)
    with pytest.raises(ValueError):
        mcm_prior_n(spec, epu.index.values[::2], epu["EPU"].to_numpy()[::2], trade.values)
