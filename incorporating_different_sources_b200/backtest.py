"""Loop level of the reference (``portfolio_calculations.py:611-658, :941-1238``) on the batched engine.

``backtest_portfolio`` keeps the reference's signature and its three output containers
(``portfolio_simple_returns_series``, ``portfolio_turnover_series``, ``portfolio_weights_metrics_df``,
consumed by ``main.py:74-91`` / ``portfolio_evaluation.py``) but evaluates ALL rebalance windows of the
backtest in one launch sequence and the whole loop body (returns, drift, turnover, cost, metrics) in one
more kernel, instead of one Python iteration per trading day (:1232-1234).

Host side = calendar / label bookkeeping only: which days rebalance (:1166-1176), which stocks form the
universe of a date and in which order (:611-658, the cap-descending ``nlargest`` order of F7).
"""
from __future__ import annotations

from datetime import timedelta
from typing import Callable, Dict, List, Optional

import numpy as np
import pandas as pd

from ._lib import SCAL
from .windows import (HF_LOOKBACK_DAYS, ffill_rows, mcm_prior_n, plan_daily_windows, plan_weekly_windows, slice_batch,
                      stack_batches, stack_windows)

# ``data_handling.extract_unique_tickers(d, d)`` of the reference reads the S&P-500 constituents of a date
# from a CSV (:619); offline there is no such file, so the universe provider is pluggable.  Default: every
# column of the market-cap frame.
UNIVERSE_PROVIDER: Optional[Callable[[pd.Timestamp], List[str]]] = None


def _tickers_for(date, stock_market_caps_df):
    if UNIVERSE_PROVIDER is not None:
        return list(UNIVERSE_PROVIDER(date))
    return list(stock_market_caps_df.columns)


def get_window_trading_days(portfolio_spec):
    mult = {"daily": 1, "weekly": 5, "monthly": 22}[portfolio_spec["rolling_window_frequency"]]
    return portfolio_spec["rolling_window"] * mult


def get_k_largest_stocks_market_caps(stock_market_caps_df, stock_prices_df, stock_intraday_prices_df, trading_date_ts,
                                     portfolio_size, rolling_window_days, rolling_window_frequency):
    """:611-658 — eligibility filter + ``nlargest(portfolio_size)`` of the caps at the trade date."""
    tickers_list = _tickers_for(trading_date_ts, stock_market_caps_df)
    if rolling_window_frequency not in HF_LOOKBACK_DAYS:
        raise RuntimeError("Unknown rolling window frequency.")                                   # :637
    days = HF_LOOKBACK_DAYS[rolling_window_frequency]
    tick = set(tickers_list)
    caps_cols = set(stock_market_caps_df.columns)
    intr_cols = set(stock_intraday_prices_df.columns)
    cand = [s for s in stock_prices_df.columns if s in tick and s in caps_cols and s in intr_cols]
    win = stock_prices_df.loc[:trading_date_ts, cand].tail(rolling_window_days)
    ok_prices = win.notna().all(axis=0)
    intr = stock_intraday_prices_df.loc[(trading_date_ts - timedelta(days=days)):(trading_date_ts + timedelta(days=1)), cand]
    ok_intr = intr.notna().any(axis=0)
    eligible = [s for s in cand if ok_prices[s] and ok_intr[s]]
    if trading_date_ts in stock_market_caps_df.index:
        daily = stock_market_caps_df.loc[trading_date_ts, eligible].dropna()
        return daily.nlargest(portfolio_size)
    raise ValueError(f"The trading date {trading_date_ts} does not exist in the market capitalizations data.")


def select_universes(stock_market_caps_df, stock_prices_df, stock_intraday_prices_df, trade_dates, portfolio_size,
                     rolling_window_days, rolling_window_frequency, lookback_days=None):
    """``get_k_largest_stocks_market_caps`` (:611-658) for ALL trade dates at once: rolling not-NaN counts of the
    daily prices (cumulative sums), per-calendar-day not-NaN counts of the intraday bars, and a stable descending
    argsort of the caps row (= ``nlargest``'s first-occurrence tie rule, F7).  Returns one ordered ticker list per
    date — membership AND order identical to the per-date function (tests/test_host_vs_reference.py).

    Also returns ``nan_bars`` [T][C] (bool, in candidate order) = the stock has a NaN bar inside the date's intraday
    LOOK-BACK of ``lookback_days`` calendar days (default: the eligibility range's own length), and the candidate list.
    Such bars do not exclude a stock: the conjugate windows drop the returns next to them, as the reference's
    ``dropna`` does (:314)."""
    if rolling_window_frequency not in HF_LOOKBACK_DAYS:
        raise RuntimeError("Unknown rolling window frequency.")                                   # :637
    days = HF_LOOKBACK_DAYS[rolling_window_frequency]
    trade_dates = pd.DatetimeIndex(trade_dates)
    T = len(trade_dates)
    caps_cols = set(stock_market_caps_df.columns)
    intr_cols = set(stock_intraday_prices_df.columns)
    cand = [s for s in stock_prices_df.columns if s in caps_cols and s in intr_cols]
    C = len(cand)
    missing = ~trade_dates.isin(stock_market_caps_df.index)
    if missing.any():
        raise ValueError(f"The trading date {trade_dates[missing][0]} does not exist in the market capitalizations data.")
    # constituents of each date (pluggable provider; default: every column)
    member = np.ones((T, C), dtype=bool)
    if UNIVERSE_PROVIDER is not None:
        pos_of = {s: j for j, s in enumerate(cand)}
        member[:] = False
        for i, d in enumerate(trade_dates):
            js = [pos_of[s] for s in UNIVERSE_PROVIDER(d) if s in pos_of]
            member[i, js] = True
    # daily prices: no NaN in the last `rolling_window_days` rows up to and including the date (:641-643)
    P = stock_prices_df[cand].to_numpy(dtype=np.float64)
    cs = np.zeros((P.shape[0] + 1, C), dtype=np.int32)
    np.cumsum(~np.isnan(P), axis=0, out=cs[1:])
    pos = stock_prices_df.index.searchsorted(trade_dates, side="right")
    lo = np.maximum(pos - int(rolling_window_days), 0)
    ok_prices = (cs[pos] - cs[lo]) == (pos - lo)[:, None]
    # intraday bars: at least one bar in [d - days, d + 1 day] (:646-647), NaN bars inside the look-back (d - D + 1d, d + 1d]
    ts = stock_intraday_prices_df.index.values.astype("datetime64[ns]")
    F = stock_intraday_prices_df[cand].to_numpy(dtype=np.float64)
    day_of = ts.astype("datetime64[D]")
    if len(ts) and (np.any(ts == day_of.astype("datetime64[ns]")) or np.any(np.diff(ts.astype(np.int64)) < 0)):
        # bars stamped exactly at midnight (or an unsorted index) do not fall into whole calendar days: per-date path
        out = [list(get_k_largest_stocks_market_caps(stock_market_caps_df, stock_prices_df, stock_intraday_prices_df, d,
                                                     portfolio_size, rolling_window_days, rolling_window_frequency).index)
               for d in trade_dates]
        return out, None, cand
    starts = np.r_[0, np.nonzero(np.diff(day_of.astype(np.int64)))[0] + 1] if len(ts) else np.zeros(0, dtype=np.int64)
    bucket_day = day_of[starts] if len(ts) else day_of
    isn = np.isnan(F)
    cnt = np.zeros((len(starts) + 1, C), dtype=np.int32)
    nanc = np.zeros((len(starts) + 1, C), dtype=np.int32)
    if len(starts):
        np.cumsum(np.add.reduceat(~isn, starts, axis=0, dtype=np.int32), axis=0, out=cnt[1:])
        np.cumsum(np.add.reduceat(isn, starts, axis=0, dtype=np.int32), axis=0, out=nanc[1:])
    d_day = trade_dates.values.astype("datetime64[D]")
    a = np.searchsorted(bucket_day, d_day - np.timedelta64(days, "D"), side="left")
    b = np.searchsorted(bucket_day, d_day, side="right")
    ok_intr = (cnt[b] - cnt[a]) > 0
    look = days if lookback_days is None else int(lookback_days)
    a_look = np.searchsorted(bucket_day, d_day - np.timedelta64(look, "D") + np.timedelta64(1, "D"), side="left")
    nan_bars = (nanc[b] - nanc[a_look]) > 0
    # caps row of each date: eligible, not NaN, k largest in first-occurrence order (:649-653)
    rows = stock_market_caps_df.index.get_indexer(trade_dates)
    V = stock_market_caps_df[cand].to_numpy(dtype=np.float64)[rows]
    valid = member & ok_prices & ok_intr & ~np.isnan(V)
    key = np.where(valid, -V, np.inf)
    order = np.argsort(key, axis=1, kind="stable")
    n_valid = valid.sum(axis=1)
    out = []
    for i in range(T):
        k = min(int(portfolio_size), int(n_valid[i]))
        out.append([cand[j] for j in order[i, :k]])
    return out, nan_bars, cand


def rebalance_flags(dates: pd.DatetimeIndex, frequency: str) -> np.ndarray:
    """Which trading days rebalance (:1166-1176): first day always; daily; Wednesday or > 7 days since the
    last rebalance; month change relative to the last rebalance."""
    flags = np.zeros(len(dates), dtype=bool)
    last = None
    for i, d in enumerate(dates):
        if last is None or frequency == "daily":
            reb = True
        elif frequency == "weekly":
            reb = d.weekday() == 2 or (d - last).days > 7
        elif frequency == "monthly":
            reb = d.month != last.month
        else:
            raise ValueError("Unknown rebalancing frequency.")                                    # :1176
        if reb:
            flags[i] = True
            last = d
    return flags


def compute_portfolio_turnover(portfolio_weights_before_df, portfolio_weights_after_df):
    """:1054-1075 — kept for API compatibility (label bookkeeping; the batched loop computes it on the device)."""
    m = portfolio_weights_before_df.merge(portfolio_weights_after_df, how="outer", left_index=True, right_index=True,
                                          suffixes=("_before", "_after")).fillna(0)
    diff = (m["Weight_before"] - m["Weight_after"]).abs().sum()
    rf_turn = abs(portfolio_weights_before_df["Weight"].sum() - portfolio_weights_after_df["Weight"].sum())
    return (diff + rf_turn) / 2


def _slice_for_date(trading_date_ts, portfolio_spec, market_data):
    """The dispatcher's slicing (:954-988)."""
    caps_all = market_data["stock_market_caps_df"]
    prices_all = market_data["stock_prices_df"]
    intr_all = market_data["stock_intraday_prices_df"]
    k = get_k_largest_stocks_market_caps(caps_all, prices_all, intr_all, trading_date_ts, portfolio_spec["size"],
                                         get_window_trading_days(portfolio_spec),
                                         portfolio_spec["rebalancing_frequency"])      # sic (:960)
    names = k.index
    caps = caps_all[names.intersection(caps_all.columns)].loc[:trading_date_ts]
    prices = prices_all[names.intersection(prices_all.columns)].loc[:trading_date_ts]
    incl = pd.Timestamp(trading_date_ts).replace(hour=23, minute=59, second=59)
    intr = intr_all[names.intersection(intr_all.columns)]
    intr = intr.loc[intr.index <= incl]
    if prices.tail(get_window_trading_days(portfolio_spec)).isna().any().any():
        raise ValueError("The filtered stock prices contain NA values.")                         # :988
    return names, caps, prices, intr


def calculate_portfolio_weights(trading_date_ts, portfolio_spec, market_data):
    """:941-1052 — per-date dispatcher for the in-scope strategies (one window per call)."""
    from . import portfolio_calculations as pc
    names, caps, prices, intr = _slice_for_date(trading_date_ts, portfolio_spec, market_data)
    rf = market_data["risk_free_rate_df"]
    strat = portfolio_spec["weighting_strategy"]
    if strat == "vw":
        return pc.calculate_value_weighted_portfolio(portfolio_spec, trading_date_ts, caps)
    if strat == "ew":
        return pc.calculate_equally_weighted_portfolio(portfolio_spec, prices)
    if strat in ("conjugate_hf_vix_vw", "conjugate_hf_vix_ew"):
        vix = market_data["vix_prices_df"]
        return pc.calculate_conjugate_hf_mcm_portfolio(portfolio_spec, trading_date_ts, caps, prices, intr,
                                                       vix.loc[vix.index <= trading_date_ts], rf)
    if strat in ("conjugate_hf_epu_vw", "conjugate_hf_epu_ew"):
        epu = market_data["epu_prices_df"]
        return pc.calculate_conjugate_hf_mcm_portfolio(portfolio_spec, trading_date_ts, caps, prices, intr,
                                                       epu.loc[epu.index <= trading_date_ts], rf)
    if strat == "jeffreys":
        return pc.calculate_jeffreys_portfolio(portfolio_spec, trading_date_ts, prices, rf)
    if strat == "jorion":
        return pc.calculate_jorion_portfolio(portfolio_spec, trading_date_ts, prices, rf)
    if strat == "shrinkage":
        return pc.calculate_shrinkage_portfolio(portfolio_spec, trading_date_ts, prices, rf)
    if strat in ("black_litterman", "greyserman"):
        raise NotImplementedError(f"strategy {strat!r} is out of scope of the CUDA path (SURVEY §2)")
    raise ValueError("Unknown weights spec.")                                                     # :1050


# HBM a stacked batch may fill: its working market (daily prices, caps and returns, intraday prices and returns) and the
# solver workspace of its windows.  The shipped spec's 178 weekly windows of 50 stocks take about 0.3 GB.
STACK_BUDGET_BYTES = 2 << 30


def _batched_weights(engine, portfolio_spec, market_data, dates_all, reb_pos, universes, hf_lookback_days=None,
                     rcond=None, counts: Optional[dict] = None):
    """Weights [R][N_all] (0 outside each date's universe) for every rebalance date.  The full market is resident in
    the engine's pool (ONE upload per backtest).  An asset set with more windows than ``engine.stack_max_windows`` gets
    its own working market -- its columns, the daily rows its windows read and their intraday look-backs, gathered on
    the device -- and one batched call.  The windows of all smaller sets (the top-k universes that change with nearly
    every rebalance date) are evaluated together instead: one stacked working market per batch of windows with the same
    number of stocks, each window in a block of its own rows and columns (``select_windows``), with the same bits as
    the per-set calls.  With the engine's condition estimate on, ``rcond`` [R] (if given) receives each window's
    estimate; vw / ew windows, which solve nothing, are left as they are.  ``counts`` (if given) receives the number
    of stacked windows and stacked calls."""
    prices_df = market_data["stock_prices_df"]
    caps_df = market_data["stock_market_caps_df"]
    intr_df = market_data["stock_intraday_prices_df"]
    rf_df = market_data["risk_free_rate_df"]
    strat = portfolio_spec["weighting_strategy"]
    all_cols = list(prices_df.columns)
    col_pos = {c: i for i, c in enumerate(all_cols)}
    N_all = len(all_cols)
    R = len(reb_pos)
    W = np.zeros((R, N_all))
    member = np.zeros((R, N_all), dtype=np.uint8)
    estimate = engine.condition_estimate and rcond is not None
    groups: Dict[tuple, List[int]] = {}
    for r, names in enumerate(universes):
        idx = tuple(sorted(col_pos[n] for n in names))
        member[r, list(idx)] = 1
        groups.setdefault(idx, []).append(r)
    dates_ns = dates_all.values.astype("datetime64[ns]")
    rf_row = ffill_rows(dates_ns, rf_df.index.values.astype("datetime64[ns]"), rf_df.iloc[:, 0].to_numpy(dtype=np.float64))
    hf_ts = intr_df.index.values.astype("datetime64[ns]")
    conj = strat.startswith("conjugate")
    needs_hf = conj or strat in ("vw", "ew")
    if portfolio_spec["rolling_window_frequency"] not in ("daily", "weekly") and strat not in ("vw", "ew"):
        raise NotImplementedError("monthly windows: resample('M') was removed from pandas (SURVEY F10)")
    if strat not in ("vw", "ew", "jeffreys", "jorion", "shrinkage") and not conj:
        raise ValueError("Unknown weights spec.")
    rf_dates = rf_df.index.values.astype("datetime64[ns]")
    rf_vals = rf_df.iloc[:, 0].to_numpy(dtype=np.float64)
    # n0 per rebalance date from the MCM series' OWN calendar (7 observations a week for FRED's EPU index; the
    # reference averages the last n observations whatever their dates, :95-112) -> injected as prior_n
    prior_n_all = None
    if conj:
        mcm_df = market_data["vix_prices_df" if "vix" in strat else "epu_prices_df"]
        prior_n_all = mcm_prior_n(portfolio_spec, mcm_df.index.values, mcm_df.iloc[:, 0].to_numpy(dtype=np.float64),
                                  dates_ns[np.asarray(reb_pos, dtype=np.int64)])
    # the whole market, once: every column, every row (intraday bars only for the strategies that read them)
    intr_cols = [c for c in all_cols if c in intr_df.columns]
    if needs_hf and len(intr_cols) != N_all:
        hf_all = intr_df.reindex(columns=all_cols).to_numpy(dtype=np.float64)
    else:
        hf_all = intr_df[all_cols].to_numpy(dtype=np.float64) if needs_hf else None
    engine.upload_pool(prices=prices_df.to_numpy(dtype=np.float64), rf_row=rf_row,
                       caps=caps_df.reindex(index=dates_all, columns=all_cols).to_numpy(dtype=np.float64), hf_prices=hf_all)
    del hf_all
    if strat in ("vw", "ew"):
        spec = dict(portfolio_spec, weighting_strategy="conjugate_hf_vix_" + strat, mcm_scaling=1,
                    rolling_window=3, rolling_window_frequency="daily", risk_aversion=1)
    else:
        spec = portfolio_spec
    stack_max = engine.stack_max_windows
    # every set's results, or the exception its planning or evaluation raised: the checks then run set by set in the
    # order of first appearance, stacked or not, so that the first failing set raises exactly as it did one by one
    outcome: Dict[tuple, object] = {}
    small = []
    for idx, rows in groups.items():
        if len(rows) <= stack_max:
            small.append((idx, rows))
            continue
        try:
            outcome[idx] = _per_set(engine, spec, strat, idx, rows, dates_ns, reb_pos, hf_ts, rf_dates, rf_vals,
                                    prior_n_all, hf_lookback_days, estimate)
        except Exception as e:          # raised below, in its set's turn
            outcome[idx] = e
    n_calls = 0
    if small:
        n_calls = _stacked_weights(engine, spec, strat, small, dates_ns, reb_pos, hf_ts, rf_dates, rf_vals, prior_n_all,
                                   hf_lookback_days, estimate, outcome)
    for idx, rows in groups.items():
        res = outcome[idx]
        if isinstance(res, Exception):
            raise res
        _store_set(strat, res, rows, list(idx), dates_all, np.asarray([reb_pos[r] for r in rows], dtype=np.int64), W,
                   rcond, estimate)
    if counts is not None:
        counts.update(stacked_windows=sum(len(rows) for _, rows in small), stacked_calls=n_calls)
    return W, member


def _plan_windows(spec, strat, dates_ns, d_idx, hf_ts, rf_dates, rf_vals, hf_lookback_days):
    """The windows of the trade-date rows ``d_idx`` on the full calendar, as both asset-set routes evaluate them:
    (ResampledRows, WindowBatch) for weekly windows, (None, WindowBatch) for daily ones.  ``spec`` is the spec the
    windows are planned with (for vw / ew the 3-price daily conjugate spec whose prior weights they read)."""
    need_hf = strat in ("vw", "ew") or strat.startswith("conjugate")
    look = hf_lookback_days if strat.startswith("conjugate") else None
    hf = hf_ts if need_hf else None
    if spec["rolling_window_frequency"] == "weekly":
        return plan_weekly_windows(spec, dates_ns, d_idx, rf_dates, rf_vals, None, hf, hf_lookback_days=look,
                                   need_hf=need_hf)
    return None, plan_daily_windows(spec, dates_ns, d_idx, hf, hf_lookback_days=look, need_hf=need_hf)


def _set_slice(batch, n_days, n_hf_rows):
    """Pool rows of one asset set's own working market (``select_market``) for a batch planned on the full calendar:
    daily windows get the rows they read and their intraday look-backs with one row in front (``hf_lo - 1``, as
    ``stack_windows`` keeps it: an empty selection is not a market), and the batch is shifted onto that slice in place;
    weekly windows keep the whole history addressable.  Returns (day_lo, day_hi, hf_lo, hf_hi)."""
    if batch.resampled:
        return 0, n_days, 0, (0 if batch.hf_lo is None else n_hf_rows)
    day_lo, day_hi = int(batch.day_row.min()) - (batch.rolling_window - 1), int(batch.day_row.max()) + 1
    batch.day_row = (batch.day_row - day_lo).astype(np.int32)
    if batch.hf_lo is None:
        return day_lo, day_hi, 0, 0
    hf_lo, hf_hi = max(int(batch.hf_lo.min()) - 1, 0), int(batch.hf_hi.max())
    batch.hf_lo = (batch.hf_lo - hf_lo).astype(np.int32)
    batch.hf_hi = (batch.hf_hi - hf_lo).astype(np.int32)
    return day_lo, day_hi, hf_lo, hf_hi


def _per_set(engine, spec, strat, idx, rows, dates_ns, reb_pos, hf_ts, rf_dates, rf_vals, prior_n_all,
             hf_lookback_days, estimate):
    """One asset set on a working market of its own: its columns, the daily rows its windows read and their intraday
    look-backs, gathered from the pool; one batched call."""
    d_idx = np.asarray([reb_pos[r] for r in rows], dtype=np.int64)
    rows_w, batch = _plan_windows(spec, strat, dates_ns, d_idx, hf_ts, rf_dates, rf_vals, hf_lookback_days)
    engine.select_market(list(idx), *_set_slice(batch, len(dates_ns), len(hf_ts)))
    if rows_w is not None:
        engine.set_resampled(rows_w)
    return _evaluate(engine, strat, batch, prior_n_all, rows, estimate)


def _evaluate(engine, strat, batch, prior_n_all, rows, estimate):
    """One batched call of the strategy on the engine's working market."""
    if strat in ("vw", "ew"):
        batch.prior_n = np.ones(batch.n_windows)                 # w0 does not depend on the MCM series
        return engine.moments(batch, outputs=("w0",))
    if strat.startswith("conjugate"):
        batch.prior_n = np.ascontiguousarray(prior_n_all[rows])
        return engine.conjugate(batch, outputs=("weights", "scalars", "status"))
    run = getattr(engine, strat)                  # jeffreys / jorion / shrinkage
    return run(batch, outputs=("weights", "status") + (("scalars",) if estimate else ()))


def _store_set(strat, res, rows, cols, dates_all, d_idx, W, rcond, estimate):
    """The checks of one asset set's windows, in the reference's order, then their weights into ``W``."""
    from . import portfolio_calculations as pc
    if strat in ("vw", "ew"):
        W[np.ix_(rows, cols)] = res["w0"]
        return
    if strat.startswith("conjugate"):
        few = np.nonzero(res["scalars"][:, SCAL["m"]] < 2)[0]
        if len(few):
            # fewer than 2 intraday returns left after dropna: the reference's S0 is all NaN (:317) and so is w1
            raise ValueError(f"conjugate_posterior_w_df contains NaN values.  ({dates_all[d_idx[few[0]]].date()}: "
                             f"{int(res['scalars'][few[0], SCAL['m']])} intraday returns left after dropping the "
                             f"missing bars)")                                            # :492-494
    _raise_on_status(res["status"], dates_all, d_idx)
    w = res["weights"]
    if estimate:
        rcond[rows] = res["scalars"][:, SCAL["rcond"]]
    if strat == "shrinkage":
        w = pc.clean_weights(w)                        # the reference returns clean_weights() (:743)
    W[np.ix_(rows, cols)] = w


def _stacked_weights(engine, spec, strat, sets, dates_ns, reb_pos, hf_ts, rf_dates, rf_vals, prior_n_all,
                     hf_lookback_days, estimate, outcome):
    """The windows of the asset sets ``sets`` [(columns, rebalance indices)], planned on the full calendar exactly as
    the per-set route plans them, relocated into stacked working markets (``stack_windows``) of one N each and
    evaluated per batch.  ``outcome[columns]`` receives each set's results, row for row as its own call would return
    them, or the exception its planning or its batch raised.  Returns the number of batched calls."""
    def plan(d):
        return _plan_windows(spec, strat, dates_ns, d, hf_ts, rf_dates, rf_vals, hf_lookback_days)

    d_of = lambda rows: np.asarray(reb_pos, dtype=np.int64)[np.asarray(rows, dtype=np.int64)]
    sets = sorted(sets, key=lambda s: len(s[0]))                          # windows of one N next to each other
    try:
        rows_w, whole = plan(np.concatenate([d_of(rows) for _, rows in sets]))
    except Exception:
        # some set cannot be planned: find which (each raises in its turn), stack the others
        ok = []
        for idx, rows in sets:
            try:
                plan(d_of(rows))
                ok.append((idx, rows))
            except Exception as e:
                outcome[idx] = e
        sets = ok
        if not sets:
            return 0
        rows_w, whole = plan(np.concatenate([d_of(rows) for _, rows in sets]))
    win_set = np.asarray([k for k, (_, rows) in enumerate(sets) for _ in rows], dtype=np.int64)
    win_r = np.asarray([r for _, rows in sets for r in rows], dtype=np.int64)
    # HBM of each window in a stack: daily blocks x (prices, caps, returns), intraday blocks x (prices, returns), solver
    stk = stack_windows(whole, rows_w)
    n_cols = np.asarray([len(sets[k][0]) for k in win_set], dtype=np.int64)
    ld, ldS = (n_cols + 15) // 16 * 16, (n_cols + 31) // 32 * 32
    hf_rows = 0 if stk.hf_lo is None else stk.hf_hi - stk.hf_lo
    nbytes = 8 * ((stk.day_hi - stk.day_lo) * 3 * ld + hf_rows * 2 * ld + (ldS + 8) * ldS + 16 * ld)
    per_window: Dict[str, list] = {}             # output name -> one row per window (the N differs between batches)
    failed: Dict[int, Exception] = {}
    n_calls = 0
    for pos in stack_batches(n_cols, nbytes, STACK_BUDGET_BYTES):
        i0, i1 = int(pos[0]), int(pos[-1]) + 1
        try:
            part = stack_windows(slice_batch(whole, i0, i1), rows_w)
            cols = np.asarray([sets[k][0] for k in win_set[i0:i1]], dtype=np.int32)
            hf = None if part.hf_lo is None else np.stack([part.hf_lo, part.hf_hi], axis=1)
            engine.select_windows(cols, np.stack([part.day_lo, part.day_hi], axis=1), hf)
            if part.resampled is not None:
                engine.set_resampled(part.resampled)
            res = _evaluate(engine, strat, part.batch, prior_n_all, win_r[i0:i1], estimate)
        except Exception as e:                  # every set with a window in this batch raises it in its turn
            for k in np.unique(win_set[i0:i1]):
                failed.setdefault(int(k), e)
            continue
        n_calls += 1
        for name, a in res.items():
            per_window.setdefault(name, [None] * len(win_r))[i0:i1] = list(a)
    for k, (idx, _) in enumerate(sets):
        if k in failed:
            outcome[idx] = failed[k]
            continue
        sel = np.nonzero(win_set == k)[0]
        outcome[idx] = {name: np.stack([rows_[i] for i in sel]) for name, rows_ in per_window.items()}
    return n_calls


def _raise_on_status(status, dates_all, d_idx):
    bad = np.nonzero(status)[0]
    if len(bad):
        raise np.linalg.LinAlgError(
            f"posterior matrix not positive definite at {dates_all[d_idx[bad[0]]].date()} "
            f"({len(bad)} of {len(d_idx)} windows): the reference's np.linalg.inv would return garbage (SURVEY F6)")


def backtest_portfolio(portfolio_spec, ts_start_date, ts_end_date, market_data, engine=None, hf_lookback_days=None,
                       timings: Optional[dict] = None, min_rcond: Optional[float] = None,
                       diagnostics: Optional[dict] = None):
    """:1221-1238 — same signature and the same three output containers.  Extensions (keyword only in spirit):
    ``engine`` (reuse a CUDA context), ``hf_lookback_days`` (the intraday look-back the reference reaches through
    ``conjugate_prior_S_df=``, e.g. 7 or 366 calendar days where its own 1-day window is rank deficient, F6),
    ``timings`` (a dict that receives the wall-clock seconds of the host / device phases, and how many windows were
    evaluated in stacked batches and in how many calls), and the condition of the
    windows: a positive-definite window with cond = 1e13 passes the pivot check and returns weights with hardly a
    correct digit.  With ``min_rcond`` or ``diagnostics`` given, every window's reciprocal 1-norm condition estimate
    (LAPACK dpocon's, from the window's own Cholesky factor, ``BayesEngine.set_condition_estimate``) is computed for
    this backtest; ``diagnostics["rcond"]`` receives it as a Series over the rebalance dates (NaN for vw / ew, which
    solve nothing), and a window below ``min_rcond`` raises ``np.linalg.LinAlgError`` naming the first such date."""
    import time
    from . import portfolio_calculations as pc
    t0 = time.perf_counter()
    eng = engine or pc._engine()
    estimate = min_rcond is not None or diagnostics is not None
    was_on = eng.condition_estimate
    if estimate:
        eng.set_condition_estimate(True)
    try:
        out, rcond = _backtest(eng, portfolio_spec, ts_start_date, ts_end_date, market_data, hf_lookback_days, timings, t0)
    finally:
        if estimate:
            eng.set_condition_estimate(was_on)
    if diagnostics is not None:
        diagnostics["rcond"] = rcond
    if min_rcond is not None:
        low = np.nonzero(rcond.to_numpy() < min_rcond)[0]
        if len(low):
            raise np.linalg.LinAlgError(
                f"ill-conditioned posterior matrix at {rcond.index[low[0]].date()} ({len(low)} of {len(rcond)} windows "
                f"with rcond below {min_rcond:g}, smallest {np.nanmin(rcond.to_numpy()):.3e}): the weights keep hardly "
                f"any correct digits")
    return out


def _backtest(eng, portfolio_spec, ts_start_date, ts_end_date, market_data, hf_lookback_days, timings, t0):
    """The body of backtest_portfolio: its three output containers and the windows' rcond Series."""
    import time
    prices_df = market_data["stock_prices_df"]
    dates_all = prices_df.index
    in_range = np.nonzero((dates_all >= ts_start_date) & (dates_all <= ts_end_date))[0]
    if len(in_range) == 0:
        raise IndexError("no trading dates in the requested range")
    bt_dates = dates_all[in_range]
    flags = rebalance_flags(bt_dates, portfolio_spec["rebalancing_frequency"])
    reb_pos = in_range[flags]
    t1 = time.perf_counter()
    universes, _, _ = select_universes(market_data["stock_market_caps_df"], prices_df,
                                                 market_data["stock_intraday_prices_df"], dates_all[reb_pos],
                                                 portfolio_spec["size"], get_window_trading_days(portfolio_spec),
                                                 portfolio_spec["rebalancing_frequency"],      # sic (:960)
                                                 lookback_days=hf_lookback_days if hf_lookback_days is not None else
                                                 HF_LOOKBACK_DAYS.get(portfolio_spec["rolling_window_frequency"]))
    t2 = time.perf_counter()
    rcond = np.full(len(reb_pos), np.nan)
    counts: dict = {}
    W, member = _batched_weights(eng, portfolio_spec, market_data, dates_all, list(reb_pos), universes, hf_lookback_days,
                                 rcond, counts)
    t3 = time.perf_counter()
    # loop body on the full column set: gathered from the resident pool, no second upload
    eng.select_market(np.arange(len(prices_df.columns)), 0, len(dates_all), 0, 0)
    scale = portfolio_spec["risk_aversion"] if portfolio_spec.get("risk_aversion") is not None else 1
    rets, turnover, metrics = eng.backtest_loop(reb_pos.astype(np.int32), W, distance_scale=scale,
                                                turnover_cost_bps=portfolio_spec["turnover_cost"],
                                                member=member, last_row=int(in_range[-1]))
    eng.upload_pool(None, None)
    name = portfolio_spec["display_name"]
    reb_dates = dates_all[reb_pos]
    returns_series = pd.Series(rets, index=bt_dates[1:], dtype="float64", name=name)
    turnover_series = pd.Series(turnover, index=reb_dates[1:], dtype="float64", name=name)
    metrics_df = pd.DataFrame(metrics, index=reb_dates, columns=["max_long", "max_short", "avg_long", "avg_short",
                                                                 "average_distance_to_comparison_portfolio"])
    if timings is not None:
        t4 = time.perf_counter()
        timings.update(calendar_s=t1 - t0, universe_selection_s=t2 - t1, weights_s=t3 - t2, loop_body_s=t4 - t3, total_s=t4 - t0,
                       rebalances=int(len(reb_pos)), asset_sets=int(len({tuple(sorted(u)) for u in universes})), **counts)
    out = {"portfolio_simple_returns_series": returns_series,
           "portfolio_turnover_series": turnover_series,
           "portfolio_weights_metrics_df": metrics_df}
    return out, pd.Series(rcond, index=reb_dates, dtype="float64", name=name)
