"""Drop-in facade: the reference's ``src/portfolio_calculations.py`` hot-path API on the B200 path.

Every function below keeps the NAME, ARGUMENT ORDER, optional-injection keywords, return container
(pandas, same labels / column names / index order) and exception types of the reference function
cited in its docstring (``:line`` = ``/root/reference/src/portfolio_calculations.py``), but the
arithmetic runs in the CUDA library (``libbayes_portfolio.so``); pandas is only used for the
label / date bookkeeping the reference also does in pandas.  There is no CPU fallback: without
the library and a B200 every call raises.

Per-window calls upload a minimal market (the window's own rows) and are meant for drop-in use and
for tests; whole backtests should use :class:`~.engine.BayesEngine` / :func:`backtest_portfolio`,
which evaluate all rebalance windows in one launch sequence.

Missing intraday bars are handled as the reference's ``dropna`` (:314-318): a NaN bar in any column of the
window drops the return rows on both sides of it (no return bridges the gap), and the realised covariance
uses the m returns that are left.  With m < 2 the prior is all NaN, as pandas' ``cov`` is, and the posterior
and portfolio functions raise the reference's ``ValueError`` (:492-494).

Deviations from the reference (documented, all raise instead of silently differing):
* ``rolling_window_frequency == "monthly"`` raises ``NotImplementedError`` (the reference itself
  fails under pandas >= 2.2, SURVEY F10);
* a window with fewer than ``rolling_window`` price rows raises ``ValueError`` (the reference would
  silently use the shorter window);
* a non-positive Cholesky pivot raises ``numpy.linalg.LinAlgError`` where ``np.linalg.inv`` would
  return garbage for a numerically singular matrix (SURVEY F6).
"""
from __future__ import annotations

import logging
from typing import Optional

import numpy as np
import pandas as pd

from ._lib import SCAL
from .windows import HF_LOOKBACK_DAYS, WindowBatch, ffill_rows, mcm_index_of, prior_kind_of

logger = logging.getLogger(__name__)
CHECK = False          # the reference's self-check flag (:30); kept for API compatibility, unused

_ENGINE = None


def _engine():
    """Module-level engine on cuda:0 (created on first use; fails loudly without a GPU)."""
    global _ENGINE
    if _ENGINE is None:
        from .engine import BayesEngine
        _ENGINE = BayesEngine(0)
    return _ENGINE


def set_engine(engine):
    """Use a caller-owned :class:`BayesEngine` (e.g. on another device)."""
    global _ENGINE
    _ENGINE = engine


# ----------------------------------------------------------------------------------------------
# window bookkeeping (pandas, as in the reference)
# ----------------------------------------------------------------------------------------------
def get_window_annualization_factor(portfolio_spec):
    """:116-124."""
    return {"daily": 252, "weekly": 52, "monthly": 12}[portfolio_spec["rolling_window_frequency"]]


def get_window_trading_days(portfolio_spec):
    """:126-134."""
    mult = {"daily": 1, "weekly": 5, "monthly": 22}[portfolio_spec["rolling_window_frequency"]]
    return portfolio_spec["rolling_window"] * mult


def _resample(df, freq):
    if freq == "daily":
        return df
    if freq == "weekly":
        return df.resample("W").last()                                   # :106, :153
    if freq == "monthly":
        raise NotImplementedError("monthly windows: resample('M') was removed from pandas (SURVEY F10)")
    raise RuntimeError("Unknown rolling window frequency.")


def adjust_stock_prices_window(portfolio_spec, trading_date_ts, k_stock_prices_df):
    """:136-161 — sort, validate the last date, optional resample, last ``rolling_window`` rows."""
    k_stock_prices_df = k_stock_prices_df.sort_index()
    if trading_date_ts != k_stock_prices_df.index[-1]:
        raise ValueError(f"trading_date_ts {trading_date_ts} must be the last date in the DataFrame.")
    win = _resample(k_stock_prices_df, portfolio_spec["rolling_window_frequency"])
    return win.iloc[-portfolio_spec["rolling_window"]:]


def _rf_rows(risk_free_rate_df, dates):
    rf_dates = risk_free_rate_df.index.values.astype("datetime64[ns]")
    rf_vals = risk_free_rate_df.iloc[:, 0].to_numpy(dtype=np.float64)
    return ffill_rows(dates, rf_dates, rf_vals)                          # :54


def _window_arrays(portfolio_spec, price_window_df, risk_free_rate_df, full_window=True):
    """Prices of one (already windowed) frame -> arrays + span + the reference's gap assertion (:40-44)."""
    n = price_window_df.shape[0]
    if full_window and n != portfolio_spec["rolling_window"]:
        raise ValueError(f"the price window has {n} rows; rolling_window={portfolio_spec['rolling_window']} "
                         "rows are required")
    if n < 3:
        raise ValueError("a window needs at least 3 price rows")
    dates = price_window_df.index.values.astype("datetime64[ns]")
    gaps = np.diff(dates).astype("timedelta64[D]").astype(np.int64)
    avg = gaps.sum() / len(gaps)
    assert gaps.max() <= avg + 4, "Unexpected large gap between return dates."    # :44
    rf_row = _rf_rows(risk_free_rate_df, dates)
    if np.isnan(rf_row).any():
        raise ValueError("risk-free rate undefined for some window dates (the reference would drop rows, :60)")
    P = np.ascontiguousarray(price_window_df.to_numpy(dtype=np.float64))
    if np.isnan(P).any():
        raise ValueError("The filtered stock prices contain NA values.")            # :988
    return P, rf_row, int(gaps.sum()), n


def _hf_window(portfolio_spec, trading_date_ts, intraday_df, columns):
    """Rows of the intraday frame inside the HF look-back (:299-312), in ``columns`` order.  NaN bars stay: the
    device drops the returns next to them (dropna, :314)."""
    freq = portfolio_spec["rolling_window_frequency"]
    if freq not in HF_LOOKBACK_DAYS:
        raise RuntimeError("Unknown rolling window frequency.")                       # :308
    D = HF_LOOKBACK_DAYS[freq]
    start = trading_date_ts - pd.Timedelta(days=D)
    idx = intraday_df.index
    sel = intraday_df[(idx > (start + pd.Timedelta(days=1))) & (idx <= (trading_date_ts + pd.Timedelta(days=1)))]
    if set(sel.columns) != set(columns):
        raise ValueError("intraday and daily price frames must hold the same stocks")
    H = np.ascontiguousarray(sel[list(columns)].to_numpy(dtype=np.float64))
    if H.shape[0] < 3:
        raise ValueError("the intraday window needs at least 3 price rows")
    return H


def _mcm_window(portfolio_spec, trading_date_ts, mcm_prices_df, n_rows):
    """Last ``rolling_window`` (resampled) MCM observations, right-aligned into ``n_rows`` slots (:90-114)."""
    mcm_prices_df = mcm_prices_df.sort_index()
    if trading_date_ts != mcm_prices_df.index[-1]:
        raise ValueError(f"trading_date_ts {trading_date_ts} must be the last date in the DataFrame.")   # :98-100
    win = _resample(mcm_prices_df, portfolio_spec["rolling_window_frequency"])
    vals = win.iloc[-portfolio_spec["rolling_window"]:].iloc[:, 0].to_numpy(dtype=np.float64)
    if np.isnan(vals).any():
        raise ValueError("NaN in the MCM window: not supported on the CUDA path")
    cnt = len(vals)
    out = np.zeros(max(n_rows, cnt))
    out[-cnt:] = vals
    return out, cnt


def _order_union(a: pd.Index, b: pd.Index) -> pd.Index:
    """Label order pandas gives ``df_a + df_b``: unchanged when equal, sorted union otherwise."""
    return a if a.equals(b) else a.union(b)


def _batch(portfolio_spec, n, span, hf_rows=None, mcm_rows=0, prior_n=None):
    strat = portfolio_spec["weighting_strategy"]
    conj = "conjugate" in strat
    return WindowBatch(
        rolling_window=n,
        day_row=np.array([n - 1], dtype=np.int32),
        span_days=np.array([span], dtype=np.int32),
        hf_lo=None if hf_rows is None else np.array([0], dtype=np.int32),
        hf_hi=None if hf_rows is None else np.array([hf_rows], dtype=np.int32),
        mcm_index=0,
        mcm_scaling=float(portfolio_spec["mcm_scaling"]) if conj and portfolio_spec.get("mcm_scaling") is not None else 1.0,
        risk_aversion=float(portfolio_spec["risk_aversion"]) if portfolio_spec.get("risk_aversion") is not None else 1.0,
        prior_weights=prior_kind_of(strat) if conj else 0,
        mcm_rows=mcm_rows,
        prior_n=None if prior_n is None else np.array([float(prior_n)]),
    )


def _upload_window(portfolio_spec, trading_date_ts, k_stock_prices_df, risk_free_rate_df,
                   k_stock_market_caps_df=None, k_stock_intraday_prices_df=None, mcm_prices_df=None,
                   prior_n=None):
    """Upload the minimal market of one window; returns (engine, batch, price columns)."""
    eng = _engine()
    win = adjust_stock_prices_window(portfolio_spec, trading_date_ts, k_stock_prices_df)
    cols = win.columns
    P, rf_row, span, n = _window_arrays(portfolio_spec, win, risk_free_rate_df)
    caps = hf = mcm = None
    hf_rows = None
    mcm_rows = 0
    if k_stock_market_caps_df is not None and "vw" in portfolio_spec["weighting_strategy"]:
        last = k_stock_market_caps_df.index[-1]
        assert last == trading_date_ts, "The last index date does not match the trading date."   # :689
        row = k_stock_market_caps_df.iloc[-1]
        if set(row.index) != set(cols):
            raise ValueError("market caps and prices must hold the same stocks")
        caps = np.zeros_like(P)
        caps[-1] = row[list(cols)].to_numpy(dtype=np.float64)
    if k_stock_intraday_prices_df is not None:
        hf = _hf_window(portfolio_spec, trading_date_ts, k_stock_intraday_prices_df, cols)
        hf_rows = hf.shape[0]
    if mcm_prices_df is not None and prior_n is None:
        m, mcm_rows = _mcm_window(portfolio_spec, trading_date_ts, mcm_prices_df, n)
        if len(m) != n:
            raise ValueError("MCM window longer than the price window")
        mcm = m[None, :]
    eng.upload_market(prices=P, rf_row=rf_row, caps=caps, hf_prices=hf, mcm=mcm)
    return eng, _batch(portfolio_spec, n, span, hf_rows, mcm_rows, prior_n), cols


def _weight_frame(values, index, index_name=None):
    df = pd.DataFrame({"Weight": np.asarray(values, dtype=np.float64)}, index=index)
    df.index.name = index_name
    return df


def _raise_no_hf_returns():
    # fewer than 2 intraday returns survive dropna: S0 is all NaN and so is w1 (:317, :492-494)
    raise ValueError("conjugate_posterior_w_df contains NaN values.")


def _check_status(status):
    if int(status) != 0:
        raise np.linalg.LinAlgError(
            f"posterior matrix is not positive definite (pivot {int(status) - 1}): the reference's "
            "np.linalg.inv would return garbage for this window (SURVEY F6)")


# ----------------------------------------------------------------------------------------------
# statistics
# ----------------------------------------------------------------------------------------------
def calculate_excess_log_returns_from_prices(portfolio_spec, stock_prices_df, risk_free_rate_df):
    """:31-62 — log returns minus the frequency-adjusted risk-free rate; first row dropped."""
    eng = _engine()
    P, rf_row, span, n = _window_arrays(portfolio_spec, stock_prices_df, risk_free_rate_df, full_window=False)
    eng.upload_market(prices=P, rf_row=rf_row)
    X = eng.excess_returns(_batch(dict(portfolio_spec, weighting_strategy="jeffreys"), n, span))
    return pd.DataFrame(X, index=stock_prices_df.index[1:], columns=stock_prices_df.columns)


def calculate_portfolio_variance(portfolio_weights_df, covariance_matrix_df):
    """:64-88 — w'Sw with both operands label-sorted."""
    w = portfolio_weights_df.sort_index()
    keys = w.index
    S = covariance_matrix_df.loc[keys, keys].to_numpy(dtype=np.float64)
    return _engine().quadratic_form(w["Weight"].to_numpy(dtype=np.float64), S)


def calculate_canonical_statistics_T(portfolio_spec, trading_date_ts, k_stock_prices_df, risk_free_rate_df):
    """:163-204 — T = X'X as an N x N frame labelled by the price columns."""
    eng, batch, cols = _upload_window(portfolio_spec, trading_date_ts, k_stock_prices_df, risk_free_rate_df)
    _, T = eng.stats(batch, want_T=True)
    return pd.DataFrame(T[0], index=cols, columns=cols)


def calculate_canonical_statistics_t(portfolio_spec, trading_date_ts, k_stock_prices_df, risk_free_rate_df):
    """:206-245 — t = column sums as an N x 1 frame (column label 0)."""
    eng, batch, cols = _upload_window(portfolio_spec, trading_date_ts, k_stock_prices_df, risk_free_rate_df)
    t, _ = eng.stats(batch, want_T=False)
    return pd.Series(t[0], index=cols).to_frame()


# ----------------------------------------------------------------------------------------------
# MCM scaling
# ----------------------------------------------------------------------------------------------
def _mcm_scalars(portfolio_spec, trading_date_ts, mcm_prices_df):
    """n0, n1, MCM average of one window from the prep kernel (dummy one-asset market)."""
    eng = _engine()
    n = portfolio_spec["rolling_window"]
    m, cnt = _mcm_window(portfolio_spec, trading_date_ts, mcm_prices_df, n)
    rows = len(m)
    spec = dict(portfolio_spec)
    if "conjugate" not in str(spec.get("weighting_strategy", "")):
        spec["weighting_strategy"] = "conjugate_hf_vix_ew"
    if spec.get("mcm_scaling") is None:
        spec["mcm_scaling"] = 1
    eng.upload_market(prices=np.ones((rows, 1)), rf_row=np.zeros(rows), caps=np.ones((rows, 1)),
                      hf_prices=np.ones((4, 1)), mcm=m[None, :])
    b = WindowBatch(rolling_window=rows, day_row=np.array([rows - 1], dtype=np.int32),
                    span_days=np.array([rows], dtype=np.int32), hf_lo=np.array([0], dtype=np.int32),
                    hf_hi=np.array([4], dtype=np.int32), mcm_index=0, mcm_scaling=float(spec["mcm_scaling"]),
                    prior_weights=1, mcm_rows=cnt)
    s = eng.moments(b, outputs=("scalars",))["scalars"][0]
    # the kernel scales by the uploaded row count; rescale to the spec's rolling_window (exact when equal)
    scale = n / rows
    return s[SCAL["n0"]] * scale, s[SCAL["mcm_avg"]]


def calculate_average_mcm_window(portfolio_spec, trading_date_ts, mcm_prices_df):
    """:90-114."""
    return float(_mcm_scalars(portfolio_spec, trading_date_ts, mcm_prices_df)[1])


def calculate_conjugate_prior_n(portfolio_spec, trading_date_ts, mcm_prices_df):
    """:247-267."""
    return float(_mcm_scalars(portfolio_spec, trading_date_ts, mcm_prices_df)[0])


def calculate_conjugate_posterior_n(portfolio_spec, trading_date_ts, mcm_prices_df, conjugate_prior_n=None):
    """:269-282."""
    if conjugate_prior_n is None:
        conjugate_prior_n = calculate_conjugate_prior_n(portfolio_spec, trading_date_ts, mcm_prices_df)
    return conjugate_prior_n + portfolio_spec["rolling_window"]


# ----------------------------------------------------------------------------------------------
# prior
# ----------------------------------------------------------------------------------------------
def calculate_conjugate_prior_S(portfolio_spec, trading_date_ts, k_stock_intraday_prices_df, mcm_prices_df,
                                conjugate_prior_n=None):
    """:285-333 — n0 * cov(h) * len(h), labelled by the intraday columns."""
    eng = _engine()
    cols = k_stock_intraday_prices_df.columns
    hf = _hf_window(portfolio_spec, trading_date_ts, k_stock_intraday_prices_df, cols)
    n = portfolio_spec["rolling_window"]
    mcm = None
    cnt = 0
    rows = 3
    if conjugate_prior_n is None:
        m, cnt = _mcm_window(portfolio_spec, trading_date_ts, mcm_prices_df, 3)
        rows = len(m)
        mcm = m[None, :]
    N = len(cols)
    eng.upload_market(prices=np.ones((rows, N)), rf_row=np.zeros(rows), caps=np.ones((rows, N)), hf_prices=hf, mcm=mcm)
    b = WindowBatch(rolling_window=rows, day_row=np.array([rows - 1], dtype=np.int32),
                    span_days=np.array([rows], dtype=np.int32), hf_lo=np.array([0], dtype=np.int32),
                    hf_hi=np.array([hf.shape[0]], dtype=np.int32), mcm_index=0,
                    mcm_scaling=float(portfolio_spec["mcm_scaling"]) * (n / rows), prior_weights=1, mcm_rows=cnt,
                    prior_n=None if conjugate_prior_n is None else np.array([float(conjugate_prior_n)]))
    _, S0 = eng.hf_cov(b)
    return pd.DataFrame(S0[0], index=cols, columns=cols)


def calculate_equally_weighted_portfolio(portfolio_spec, k_stock_prices_df):
    """:661-677 — 1/size for every price column; index name 'Stock'."""
    num = portfolio_spec["size"]
    cols = k_stock_prices_df.columns
    eng = _engine()
    N = len(cols)
    eng.upload_market(prices=np.ones((3, N)), rf_row=np.zeros(3), caps=np.ones((3, N)), hf_prices=np.ones((4, N)),
                      mcm=np.ones((1, 3)))
    b = WindowBatch(rolling_window=3, day_row=np.array([2], dtype=np.int32), span_days=np.array([3], dtype=np.int32),
                    hf_lo=np.array([0], dtype=np.int32), hf_hi=np.array([4], dtype=np.int32), prior_weights=1)
    w0 = eng.moments(b, outputs=("w0",))["w0"][0]
    if num != N:
        # the reference builds [1/size]*size against the frame's columns and raises on a length mismatch
        raise ValueError(f"Length of values ({num}) does not match length of index ({N})")
    return _weight_frame(w0, cols, "Stock")


def calculate_value_weighted_portfolio(portfolio_spec, trading_date_ts, k_stock_market_caps_df):
    """:679-701 — caps of the last row, sorted descending, normalised; index name 'Stock'."""
    series = k_stock_market_caps_df.iloc[-1].sort_values(ascending=False)
    last = k_stock_market_caps_df.index[-1]
    assert last == trading_date_ts, "The last index date does not match the trading date."   # :689
    eng = _engine()
    N = len(series)
    caps = np.ones((3, N))
    caps[-1] = series.to_numpy(dtype=np.float64)
    eng.upload_market(prices=np.ones((3, N)), rf_row=np.zeros(3), caps=caps, hf_prices=np.ones((4, N)),
                      mcm=np.ones((1, 3)))
    b = WindowBatch(rolling_window=3, day_row=np.array([2], dtype=np.int32), span_days=np.array([3], dtype=np.int32),
                    hf_lo=np.array([0], dtype=np.int32), hf_hi=np.array([4], dtype=np.int32), prior_weights=0)
    w0 = eng.moments(b, outputs=("w0",))["w0"][0]
    return _weight_frame(w0, series.index, "Stock")


def calculate_conjugate_prior_w(portfolio_spec, trading_date_ts, k_stock_prices_df, k_stock_market_caps_df,
                                mcm_prices_df):
    """:361-380."""
    if "vw" in portfolio_spec["weighting_strategy"]:
        return calculate_value_weighted_portfolio(portfolio_spec, trading_date_ts, k_stock_market_caps_df)
    if "ew" in portfolio_spec["weighting_strategy"]:
        return calculate_equally_weighted_portfolio(portfolio_spec, k_stock_prices_df)
    raise ValueError("Unknown conjugate portfolio prior weights.")


# ----------------------------------------------------------------------------------------------
# conjugate posterior
# ----------------------------------------------------------------------------------------------
def _conj_fused(portfolio_spec, trading_date_ts, k_stock_prices_df, k_stock_market_caps_df,
                k_stock_intraday_prices_df, mcm_prices_df, risk_free_rate_df, outputs, solve):
    eng, batch, cols = _upload_window(portfolio_spec, trading_date_ts, k_stock_prices_df, risk_free_rate_df,
                                      k_stock_market_caps_df, k_stock_intraday_prices_df, mcm_prices_df)
    if solve:
        res = eng.conjugate(batch, outputs=tuple(outputs) + ("scalars", "status"))
        if res["scalars"][0][SCAL["m"]] < 2:
            _raise_no_hf_returns()
        _check_status(res["status"][0])
    else:
        res = eng.moments(batch, outputs=tuple(outputs))
    order = _order_union(k_stock_intraday_prices_df.columns, cols)
    return res, cols, order


def _reorder(vec_or_mat, cols, order):
    pos = cols.get_indexer(order)
    a = np.asarray(vec_or_mat)
    return a[pos] if a.ndim == 1 else a[np.ix_(pos, pos)]


def calculate_conjugate_posterior_S(portfolio_spec, trading_date_ts, k_stock_prices_df, k_stock_intraday_prices_df,
                                    mcm_prices_df, risk_free_rate_df, conjugate_prior_S_df=None):
    """:335-358 — S1 = S0 + T."""
    if conjugate_prior_S_df is None:
        spec = dict(portfolio_spec)
        if "vw" in spec["weighting_strategy"]:
            spec["weighting_strategy"] = spec["weighting_strategy"].replace("vw", "ew")   # S1 does not need caps
        res, cols, order = _conj_fused(spec, trading_date_ts, k_stock_prices_df, None, k_stock_intraday_prices_df,
                                       mcm_prices_df, risk_free_rate_df, ("S1",), solve=False)
        return pd.DataFrame(_reorder(res["S1"][0], cols, order), index=order, columns=order)
    T_df = calculate_canonical_statistics_T(portfolio_spec, trading_date_ts, k_stock_prices_df, risk_free_rate_df)
    order = _order_union(conjugate_prior_S_df.columns, T_df.columns)
    S0 = conjugate_prior_S_df.loc[order, order].to_numpy(dtype=np.float64)
    T = T_df.loc[order, order].to_numpy(dtype=np.float64)
    N = len(order)
    res = _engine().dense_posterior(jeffreys=False, rolling_window=portfolio_spec["rolling_window"], risk_aversion=1.0,
                                    T=T, t=np.zeros(N), S0=S0, w0=np.full(N, 1.0 / N), n0=1.0, c=1.0)
    return pd.DataFrame(res["S1"], index=order, columns=order)


def calculate_conjugate_c(portfolio_spec, trading_date_ts, k_stock_prices_df, k_stock_market_caps_df,
                          k_stock_intraday_prices_df, mcm_prices_df, conjugate_prior_n=None,
                          conjugate_prior_S_df=None, conjugate_prior_w_df=None):
    """:382-430 — c = 2 n0 / ((n0+N+2) + sqrt((n0+N+2)^2 + 4 n0 w0'S0w0))."""
    if conjugate_prior_n is None:
        conjugate_prior_n = calculate_conjugate_prior_n(portfolio_spec, trading_date_ts, mcm_prices_df)
    if conjugate_prior_S_df is None:
        conjugate_prior_S_df = calculate_conjugate_prior_S(portfolio_spec, trading_date_ts,
                                                           k_stock_intraday_prices_df, mcm_prices_df)
    if conjugate_prior_w_df is None:
        conjugate_prior_w_df = calculate_conjugate_prior_w(portfolio_spec, trading_date_ts, k_stock_prices_df,
                                                           k_stock_market_caps_df, mcm_prices_df)
    w = conjugate_prior_w_df.sort_index()
    keys = w.index
    S0 = conjugate_prior_S_df.loc[keys, keys].to_numpy(dtype=np.float64)
    if len(keys) != portfolio_spec["size"]:
        logger.warning("conjugate_c: %d assets but spec size %d", len(keys), portfolio_spec["size"])
    res = _engine().dense_posterior(jeffreys=False, rolling_window=portfolio_spec["rolling_window"], risk_aversion=1.0,
                                    T=None, t=None, S0=S0, w0=w["Weight"].to_numpy(dtype=np.float64),
                                    n0=float(conjugate_prior_n))
    c = float(res["scalars"][SCAL["c"]])
    if len(keys) != portfolio_spec["size"]:
        # the reference uses spec["size"], not the frame width, inside the formula (:415-416)
        v0 = float(res["scalars"][SCAL["v0"]])
        k = conjugate_prior_n + portfolio_spec["size"] + 2
        c = (2 * conjugate_prior_n) / (k + (k ** 2 + 4 * conjugate_prior_n * v0) ** 0.5)
    return c


def _dense_conjugate(portfolio_spec, trading_date_ts, k_stock_prices_df, k_stock_market_caps_df,
                     k_stock_intraday_prices_df, mcm_prices_df, risk_free_rate_df, conjugate_c=None,
                     conjugate_prior_n=None, conjugate_posterior_n=None, conjugate_prior_S_df=None,
                     conjugate_posterior_S_df=None, conjugate_prior_w_df=None, conjugate_posterior_w_df=None):
    """Staged path used whenever a moment is injected: missing pieces come from the fused kernels."""
    need_n0 = conjugate_c is None or (conjugate_posterior_n is None)
    if conjugate_prior_n is None and need_n0:
        conjugate_prior_n = calculate_conjugate_prior_n(portfolio_spec, trading_date_ts, mcm_prices_df)
    if conjugate_prior_S_df is None:
        conjugate_prior_S_df = calculate_conjugate_prior_S(portfolio_spec, trading_date_ts, k_stock_intraday_prices_df,
                                                           mcm_prices_df, conjugate_prior_n=conjugate_prior_n)
    if conjugate_prior_w_df is None:
        conjugate_prior_w_df = calculate_conjugate_prior_w(portfolio_spec, trading_date_ts, k_stock_prices_df,
                                                           k_stock_market_caps_df, mcm_prices_df)
    eng, batch, cols = _upload_window(portfolio_spec, trading_date_ts, k_stock_prices_df, risk_free_rate_df)
    t, T = eng.stats(batch, want_T=True)
    S1_order = (conjugate_posterior_S_df.columns if conjugate_posterior_S_df is not None
                else _order_union(conjugate_prior_S_df.columns, cols))
    pos = cols.get_indexer(S1_order)
    if (pos < 0).any() or len(S1_order) != len(cols):
        raise ValueError("posterior S and prices must hold the same stocks")
    kw = dict(
        T=T[0][np.ix_(pos, pos)], t=t[0][pos],
        S0=conjugate_prior_S_df.loc[S1_order, S1_order].to_numpy(dtype=np.float64),
        w0=conjugate_prior_w_df["Weight"].reindex(S1_order).to_numpy(dtype=np.float64),
        n0=float(conjugate_prior_n) if conjugate_prior_n is not None else 0.0,
        n1=conjugate_posterior_n, c=conjugate_c,
        S1=None if conjugate_posterior_S_df is None else conjugate_posterior_S_df.loc[S1_order, S1_order].to_numpy(dtype=np.float64),
        w1=None if conjugate_posterior_w_df is None else conjugate_posterior_w_df["Weight"].reindex(S1_order).to_numpy(dtype=np.float64),
    )
    gamma = portfolio_spec["risk_aversion"] if portfolio_spec.get("risk_aversion") is not None else 1.0
    res = eng.dense_posterior(jeffreys=False, rolling_window=portfolio_spec["rolling_window"], risk_aversion=gamma, **kw)
    if conjugate_posterior_w_df is None:
        if np.isnan(kw["S0"]).any():
            _raise_no_hf_returns()
        _check_status(res["status"][0])
    return res, S1_order


def calculate_conjugate_posterior_w(portfolio_spec, trading_date_ts, k_stock_prices_df, k_stock_market_caps_df,
                                    k_stock_intraday_prices_df, mcm_prices_df, risk_free_rate_df, conjugate_c=None,
                                    conjugate_prior_w_df=None, conjugate_prior_S_df=None,
                                    conjugate_posterior_S_df=None):
    """:432-496 — w1 = S1^-1 (c S0 w0 + t)."""
    injected = any(x is not None for x in (conjugate_c, conjugate_prior_w_df, conjugate_prior_S_df,
                                           conjugate_posterior_S_df))
    if not injected:
        res, cols, order = _conj_fused(portfolio_spec, trading_date_ts, k_stock_prices_df, k_stock_market_caps_df,
                                       k_stock_intraday_prices_df, mcm_prices_df, risk_free_rate_df, ("w1",), True)
        w1 = _reorder(res["w1"][0], cols, order)
    else:
        res, order = _dense_conjugate(portfolio_spec, trading_date_ts, k_stock_prices_df, k_stock_market_caps_df,
                                      k_stock_intraday_prices_df, mcm_prices_df, risk_free_rate_df,
                                      conjugate_c=conjugate_c, conjugate_prior_S_df=conjugate_prior_S_df,
                                      conjugate_posterior_S_df=conjugate_posterior_S_df,
                                      conjugate_prior_w_df=conjugate_prior_w_df)
        w1 = res["w1"]
    if np.isnan(w1).any():
        raise ValueError("conjugate_posterior_w_df contains NaN values.")                      # :492-494
    return _weight_frame(w1, order)


def calculate_mean_conjugate_posterior_nu(portfolio_spec, trading_date_ts, k_stock_prices_df, k_stock_market_caps_df,
                                          k_stock_intraday_prices_df, mcm_prices_df, risk_free_rate_df,
                                          conjugate_c=None, conjugate_prior_n=None, conjugate_posterior_n=None,
                                          conjugate_prior_S_df=None, conjugate_posterior_S_df=None,
                                          conjugate_prior_w_df=None, conjugate_posterior_w_df=None):
    """:499-577 — nu = (n1 + N + 2) w1 / (n1 - w1'S1w1)."""
    injected = any(x is not None for x in (conjugate_c, conjugate_prior_n, conjugate_posterior_n, conjugate_prior_S_df,
                                           conjugate_posterior_S_df, conjugate_prior_w_df, conjugate_posterior_w_df))
    if not injected:
        res, cols, order = _conj_fused(portfolio_spec, trading_date_ts, k_stock_prices_df, k_stock_market_caps_df,
                                       k_stock_intraday_prices_df, mcm_prices_df, risk_free_rate_df, ("nu",), True)
        nu = _reorder(res["nu"][0], cols, order)
    else:
        res, order = _dense_conjugate(portfolio_spec, trading_date_ts, k_stock_prices_df, k_stock_market_caps_df,
                                      k_stock_intraday_prices_df, mcm_prices_df, risk_free_rate_df,
                                      conjugate_c=conjugate_c, conjugate_prior_n=conjugate_prior_n,
                                      conjugate_posterior_n=conjugate_posterior_n,
                                      conjugate_prior_S_df=conjugate_prior_S_df,
                                      conjugate_posterior_S_df=conjugate_posterior_S_df,
                                      conjugate_prior_w_df=conjugate_prior_w_df,
                                      conjugate_posterior_w_df=conjugate_posterior_w_df)
        nu = res["nu"]
    return _weight_frame(nu, order)


def calculate_mean_jeffreys_posterior_nu(portfolio_spec, trading_date_ts, k_stock_prices_df, risk_free_rate_df):
    """:580-608 — (T - t t'/n)^-1 t, column renamed 'Weight'."""
    eng, batch, cols = _upload_window(dict(portfolio_spec, weighting_strategy="jeffreys"), trading_date_ts,
                                      k_stock_prices_df, risk_free_rate_df)
    res = eng.jeffreys(batch, outputs=("nu", "status"))
    _check_status(res["status"][0])
    return _weight_frame(res["nu"][0], cols)


# ----------------------------------------------------------------------------------------------
# weight functions (the drop-in boundary proper, :819-849)
# ----------------------------------------------------------------------------------------------
def calculate_conjugate_hf_mcm_portfolio(portfolio_spec, trading_date_ts, k_stock_market_caps_df, k_stock_prices_df,
                                         k_stock_intraday_prices_df, mcm_prices_df, risk_free_rate_df):
    """:819-836 — (1/gamma) * nu, one launch sequence (prep, fused Gram, Cholesky solve)."""
    res, cols, order = _conj_fused(portfolio_spec, trading_date_ts, k_stock_prices_df, k_stock_market_caps_df,
                                   k_stock_intraday_prices_df, mcm_prices_df, risk_free_rate_df, ("weights",), True)
    return _weight_frame(_reorder(res["weights"][0], cols, order), order)


def calculate_jeffreys_portfolio(portfolio_spec, trading_date_ts, k_stock_prices_df, risk_free_rate_df):
    """:838-849."""
    eng, batch, cols = _upload_window(dict(portfolio_spec, weighting_strategy="jeffreys"), trading_date_ts,
                                      k_stock_prices_df, risk_free_rate_df)
    res = eng.jeffreys(batch, outputs=("weights", "status"))
    _check_status(res["status"][0])
    return _weight_frame(res["weights"][0], cols)


# ----------------------------------------------------------------------------------------------
# sibling estimators on the same sample moments (SURVEY §8(f) rank 3, :703-758, :851-895)
# ----------------------------------------------------------------------------------------------
def calculate_jorion_portfolio(portfolio_spec, trading_date_ts, k_stock_prices_df, risk_free_rate_df):
    """:851-895 — Jorion's Bayes-Stein portfolio; index named 'Stock' as in the reference (:893)."""
    N = len(k_stock_prices_df.columns)
    if portfolio_spec["rolling_window"] - 1 - N - 2 <= 0:
        raise ValueError("Jorion needs T - N - 2 > 0 (T = rolling_window - 1 returns, :879)")
    eng, batch, cols = _upload_window(dict(portfolio_spec, weighting_strategy="jeffreys"), trading_date_ts,
                                      k_stock_prices_df, risk_free_rate_df)
    res = eng.jorion(batch, outputs=("weights", "status"))
    _check_status(res["status"][0])
    return _weight_frame(res["weights"][0], cols, index_name="Stock")


def clean_weights(weights, cutoff=1e-4, rounding=5):
    """pypfopt 1.5.5 ``base_optimizer.clean_weights``: |w| < cutoff -> 0, then round (called at :743)."""
    w = np.array(weights, dtype=np.float64, copy=True)
    w[np.abs(w) < cutoff] = 0.0
    return np.round(w, rounding)


def calculate_shrinkage_portfolio(portfolio_spec, trading_date_ts, k_stock_prices_df, risk_free_rate_df,
                                  clean=True):
    """:703-758 — Ledoit-Wolf shrinkage tangency weights, index named 'Stock' (:744).

    The reference obtains them from a cvxpy solve (pypfopt ``EfficientFrontier.max_quadratic_utility`` with a
    zero-variance RISK_FREE column and inactive bounds) and checks them against ``(1/gamma) Sigma^-1 mu`` to
    1e-4 (:748-756); the device computes that closed form directly and ``clean=True`` applies the
    ``clean_weights()`` cutoff / 5-decimal rounding the reference returns (:743).  pypfopt and cvxpy are not
    installed here, so parity of this function is pinned against sklearn's ``ledoit_wolf`` (what pypfopt calls)
    on the reference's own excess returns, not against the reference's rounded solver output."""
    eng, batch, cols = _upload_window(dict(portfolio_spec, weighting_strategy="jeffreys"), trading_date_ts,
                                      k_stock_prices_df, risk_free_rate_df)
    res = eng.shrinkage(batch, outputs=("weights", "status"))
    _check_status(res["status"][0])
    w = res["weights"][0]
    return _weight_frame(clean_weights(w) if clean else w, cols, index_name="Stock")


# ----------------------------------------------------------------------------------------------
# loop level (:611-658, :941-1238): see backtest.py
# ----------------------------------------------------------------------------------------------
from .backtest import (  # noqa: E402,F401
    backtest_portfolio,
    calculate_portfolio_weights,
    compute_portfolio_turnover,
    get_k_largest_stocks_market_caps,
    rebalance_flags,
)
