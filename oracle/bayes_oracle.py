"""TEST INFRASTRUCTURE — CPU oracle for the Bayesian tangency-weight hot path.

A plain NumPy restatement of the arithmetic in the reference's
``src/portfolio_calculations.py`` (all ``:line`` citations below are into that
file).  It exists to CHECK the CUDA path; it is never the thing shipped or
measured: only ``tests/``, ``__graft_entry__.smoke()`` and the ``cpu_baseline`` /
``--impl reference`` legs of ``bench.py`` may import it.

Parity pinning: the reference ships no tests, golden vectors or fixtures for this
path (SURVEY.md §4, §8(c)), so the oracle is pinned against *the reference itself
executed in the build container* (NumPy 2.3.5 / pandas 3.0.2) on seeded synthetic
markets: ``tests/golden/make_golden.py`` runs the unmodified reference (through
``oracle/ref_import.py``) and commits its outputs under ``tests/golden/``;
``tests/test_oracle_golden.py`` checks this file against those vectors to 1e-12.

Conventions: a "market" is any object with NumPy attributes ``dates`` (D,
datetime64[ns]), ``prices`` / ``caps`` (D, N), ``hf_ts`` (R, datetime64[ns]),
``hf_prices`` (R, N), ``vix`` / ``epu`` / ``rf`` (D,) — see
``incorporating_different_sources_b200/synthetic.py``.  ``cols`` is the ordered
list of asset columns of one window (cap-descending at the trade date, F7).
Third-party arithmetic the reference delegates to (not vendored there): NumPy
``np.log`` / ``np.dot`` / ``np.cov`` / ``np.linalg.inv`` (requirements.txt pins
numpy==1.24.4; this container has 2.3.5) — called here exactly where the
reference calls them.
"""
from __future__ import annotations

import numpy as np

_DAY = np.timedelta64(1, "D")
HF_LOOKBACK_DAYS = {"daily": 1, "weekly": 7, "monthly": 31}   # :299-304


# --------------------------------------------------------------------------- windows
def _week_id(dates_ns: np.ndarray) -> np.ndarray:
    """Week bucket of ``resample('W')`` (weeks end on Sunday).  1970-01-01 is a Thursday."""
    days = dates_ns.astype("datetime64[D]").astype(np.int64)
    return (days + 3) // 7


def _week_label(week_id: np.ndarray) -> np.ndarray:
    """Sunday that closes the bucket — the label ``resample('W').last()`` assigns (:153)."""
    return ((week_id * 7 + 3).astype("datetime64[D]")).astype("datetime64[ns]")


def resample_weekly_last(dates: np.ndarray, values: np.ndarray):
    """``df.resample('W').last()`` for a NaN-free frame without empty weeks (:106,:153)."""
    wid = _week_id(dates)
    if np.any(np.diff(wid) > 1):
        raise NotImplementedError("empty week in resample('W'): the reference would emit a NaN row")
    last = np.r_[np.nonzero(np.diff(wid))[0], len(wid) - 1]
    return _week_label(wid[last]), values[last], last


def adjust_stock_prices_window(spec, dates, prices, d):
    """:136-161 — validate last date, optional weekly resample, last ``rolling_window`` rows.

    ``dates``/``prices`` must already be truncated to rows <= d (the dispatcher does
    that at :969).  Returns (window_dates, window_prices).
    """
    if dates[-1] != d:
        raise ValueError(f"trading_date_ts {d} must be the last date in the DataFrame.")   # :145-147
    n = spec["rolling_window"]
    freq = spec["rolling_window_frequency"]
    if freq == "daily":
        wd, wp = dates, prices
    elif freq == "weekly":
        wd, wp, _ = resample_weekly_last(dates, prices)
    else:
        raise NotImplementedError("monthly windows: resample('M') no longer exists in pandas 3 (SURVEY F10)")
    return wd[-n:], wp[-n:]


def excess_log_returns(win_dates, win_prices, rf_dates, rf_values):
    """:31-62 — log returns minus the per-window frequency-adjusted risk-free rate."""
    logret = np.log(win_prices[1:] / win_prices[:-1])                                   # :37
    gaps = np.diff(win_dates).astype("timedelta64[D]").astype(np.int64)                 # :40
    avg = gaps.sum() / len(gaps)                                                        # :41
    assert gaps.max() <= avg + 4, "Unexpected large gap between return dates."          # :44
    adj = (1 + rf_values) ** (avg / 365) - 1                                            # :48
    idx = np.searchsorted(rf_dates, win_dates, side="right") - 1                        # :54 ffill
    if np.any(idx < 0):
        raise ValueError("risk-free series starts after the window (NaN rows would be dropped, :60)")
    a = adj[idx][1:]                                                                    # first row is NaN, :60
    return logret - a[:, None]                                                          # :57


def canonical_T(X):
    return np.dot(X.T, X)                                                               # :180-182


def canonical_t(X):
    return X.sum(axis=0)                                                                # :222


# --------------------------------------------------------------------------- MCM
def average_mcm_window(spec, mcm_dates, mcm_values, d):
    """:90-114 — mean of the last ``rolling_window`` (resampled) MCM observations incl. d."""
    if mcm_dates[-1] != d:
        raise ValueError(f"trading_date_ts {d} must be the last date in the DataFrame.")   # :98-100
    freq = spec["rolling_window_frequency"]
    if freq == "daily":
        v = mcm_values
    elif freq == "weekly":
        _, v, _ = resample_weekly_last(mcm_dates, mcm_values)
    else:
        raise NotImplementedError("monthly")
    return float(np.mean(v[-spec["rolling_window"]:]))                                  # :112


def conjugate_prior_n(spec, mcm_dates, mcm_values, d):
    """:247-267."""
    avg = average_mcm_window(spec, mcm_dates, mcm_values, d)
    cur = float(mcm_values[-1])                                                         # :257 (last row == d)
    frac = cur / avg if cur > avg else avg / cur                                        # :260-263
    return spec["rolling_window"] * frac * spec["mcm_scaling"]                          # :265


def conjugate_posterior_n(spec, n0):
    return n0 + spec["rolling_window"]                                                  # :282


# --------------------------------------------------------------------------- HF prior
def hf_window_rows(spec, hf_ts, d, lookback_days=None):
    """Row range [lo, hi) of intraday prices with ``d-D+1d < ts <= d+1d`` (:310-312).

    ``lookback_days`` overrides the reference's table {daily:1, weekly:7, monthly:31}
    (:299-304); the reference reaches other look-backs only through the
    ``conjugate_prior_S_df=`` injection parameter (SURVEY F5).
    """
    if lookback_days is None:
        freq = spec["rolling_window_frequency"]
        if freq not in HF_LOOKBACK_DAYS:
            raise RuntimeError("Unknown rolling window frequency.")                    # :308
        lookback_days = HF_LOOKBACK_DAYS[freq]
    start = d - lookback_days * _DAY + _DAY
    lo = int(np.searchsorted(hf_ts, start, side="right"))
    hi = int(np.searchsorted(hf_ts, d + _DAY, side="right"))
    return lo, hi


def realized_covariance(hf_prices_window):
    """:314-318 — ``cov(h) * len(h)``: demeaned, ddof=1, re-scaled by m (SURVEY F4)."""
    h = np.log(hf_prices_window[1:] / hf_prices_window[:-1])                            # :314
    m = h.shape[0]
    return np.cov(h.T) * m, m                                                           # :317-318


def conjugate_prior_S(n0, hf_prices_window):
    rc, _ = realized_covariance(hf_prices_window)
    return n0 * rc                                                                      # :333


# --------------------------------------------------------------------------- weights
def prior_w(spec, caps_row):
    """:361-380 → :679-701 (value weighted) / :661-677 (equally weighted)."""
    strat = spec["weighting_strategy"]
    if "vw" in strat:
        return caps_row / caps_row.sum()                                                # :692-695
    if "ew" in strat:
        return np.full(spec["size"], 1 / spec["size"])                                  # :670-672
    raise ValueError("Unknown conjugate portfolio prior weights.")                      # :378


def portfolio_variance(w, S):
    return float(np.dot(w.T, np.dot(S, w)))                                             # :78


def conjugate_c(spec, n0, S0, w0):
    """:415-418."""
    k = n0 + spec["size"] + 2
    return (2 * n0) / (k + (k ** 2 + 4 * n0 * portfolio_variance(w0, S0)) ** (1 / 2))


def conjugate_posterior_w(c, S0, w0, S1, t):
    """:485-489 — explicit inverse, then mat-vec."""
    S1_inv = np.linalg.inv(S1)
    w1 = np.dot(S1_inv, c * np.dot(S0, w0) + t)
    if np.isnan(w1).any():
        raise ValueError("conjugate_posterior_w_df contains NaN values.")               # :492-494
    return w1


def mean_conjugate_posterior_nu(spec, n1, w1, S1):
    """:572-575."""
    return (n1 + spec["size"] + 2) * w1 / (n1 - portfolio_variance(w1, S1))


def mean_jeffreys_posterior_nu(spec, T, t):
    """:600-606 — note the division by ``rolling_window`` (prices), not n-1 returns (F2)."""
    J = T - 1 / spec["rolling_window"] * np.outer(t, t)
    return np.dot(np.linalg.inv(J), t), J


# --------------------------------------------------------------------------- per-window drivers
def _mcm_series(spec, mkt):
    strat = spec["weighting_strategy"]
    if "vix" in strat:
        return mkt.vix
    if "epu" in strat:
        return mkt.epu
    raise ValueError("Unknown weights spec.")                                           # :1050


def daily_statistics(spec, mkt, d_idx, cols):
    d = mkt.dates[d_idx]
    wd, wp = adjust_stock_prices_window(spec, mkt.dates[: d_idx + 1], mkt.prices[: d_idx + 1][:, cols], d)
    rf_dates = getattr(mkt, "rf_dates", mkt.dates)
    X = excess_log_returns(wd, wp, rf_dates, mkt.rf)
    return canonical_t(X), canonical_T(X), X


def conjugate_window(spec, mkt, d_idx, cols, hf_lookback_days=None):
    """``calculate_conjugate_hf_mcm_portfolio`` (:819-836) with every posterior moment exposed."""
    cols = np.asarray(cols)
    d = mkt.dates[d_idx]
    N = spec["size"]
    t, T, _ = daily_statistics(spec, mkt, d_idx, cols)
    mcm = _mcm_series(spec, mkt)
    n0 = conjugate_prior_n(spec, mkt.dates[: d_idx + 1], mcm[: d_idx + 1], d)
    n1 = conjugate_posterior_n(spec, n0)
    lo, hi = hf_window_rows(spec, mkt.hf_ts, d, hf_lookback_days)
    rc, m = realized_covariance(mkt.hf_prices[lo:hi][:, cols])
    S0 = n0 * rc
    w0 = prior_w(spec, mkt.caps[d_idx, cols])
    v0 = portfolio_variance(w0, S0)
    c = conjugate_c(spec, n0, S0, w0)
    S1 = S0 + T                                                                         # :358
    w1 = conjugate_posterior_w(c, S0, w0, S1, t)
    v1 = portfolio_variance(w1, S1)
    nu = mean_conjugate_posterior_nu(spec, n1, w1, S1)
    weights = 1 / spec["risk_aversion"] * nu                                            # :836
    return dict(t=t, T=T, n0=n0, n1=n1, S0=S0, S1=S1, w0=w0, v0=v0, c=c, w1=w1, v1=v1,
                nu=nu, weights=weights, hf_returns=m, N=N)


def jeffreys_window(spec, mkt, d_idx, cols):
    """``calculate_jeffreys_portfolio`` (:838-849)."""
    cols = np.asarray(cols)
    t, T, _ = daily_statistics(spec, mkt, d_idx, cols)
    nu, J = mean_jeffreys_posterior_nu(spec, T, t)
    weights = 1 / spec["risk_aversion"] * nu                                            # :849
    return dict(t=t, T=T, J=J, nu=nu, weights=weights)


# --------------------------------------------------------------------------- sibling estimators (SURVEY 8(f) rank 3)
def jorion_window(spec, mkt, d_idx, cols):
    """``calculate_jorion_portfolio`` (:851-895): Bayes-Stein shrinkage, explicit inverses as in the reference."""
    cols = np.asarray(cols)
    t, T_stat, X = daily_statistics(spec, mkt, d_idx, cols)
    N = len(cols)                                                                       # :869
    T = len(X)                                                                          # :870
    mu_hat = X.mean(axis=0)                                                             # :873
    V_hat = np.cov(X, rowvar=False)                                                     # :876 (ddof = 1)
    V_bar = T / (T - N - 2) * V_hat                                                     # :879
    V_bar_inv = np.linalg.inv(V_bar)                                                    # :880
    one = np.ones(N)
    one_vinv_one = np.dot(np.dot(one, V_bar_inv), one)
    mu_g = np.dot(np.dot(one, V_bar_inv), mu_hat) / one_vinv_one                        # :882
    diff = mu_hat - mu_g * one                                                          # :884
    q = np.dot(np.dot(diff, V_bar_inv), diff)
    lam = (N + 2) / q                                                                   # :885
    v_hat = (N + 2) / ((N + 2) + T * q)                                                 # :887
    V_PJ = (1 + 1 / (T + lam)) * V_bar + lam / (T * (T + 1 + lam)) * np.outer(one, one) / one_vinv_one   # :888
    mu_PJ = (1 - v_hat) * mu_hat + v_hat * mu_g * one                                   # :889
    weights = 1 / spec["risk_aversion"] * np.dot(np.linalg.inv(V_PJ), mu_PJ)            # :891-893
    return dict(t=t, mu_hat=mu_hat, V_hat=V_hat, mu_g=mu_g, q=q, lambda_hat=lam, v_hat=v_hat,
                one_vinv_one=one_vinv_one, weights=weights)


def ledoit_wolf(X):
    """``sklearn.covariance.ledoit_wolf(X)`` (scikit-learn >= 0.24 ``_shrunk_covariance.py``: ``ledoit_wolf_shrinkage``
    + ``_ledoit_wolf``), the routine pypfopt 1.5.5 ``CovarianceShrinkage.ledoit_wolf()`` (constant-variance target)
    calls on the returns at :727-729.  pypfopt and its call site cannot run here (not installed); this restatement is
    pinned against the installed sklearn in ``tests/test_oracle_golden.py``.  Returns (shrunk_cov, shrinkage)."""
    n_samples, n_features = X.shape
    Xc = X - X.mean(0)
    if n_features == 1:           # sklearn's one-feature rule: "the result is the same whatever the shrinkage"
        return np.atleast_2d((Xc ** 2).mean()), 0.0
    X2 = Xc ** 2
    emp_cov_trace = np.sum(X2, axis=0) / n_samples
    mu = np.sum(emp_cov_trace) / n_features
    beta_ = np.sum(np.dot(X2.T, X2))
    delta_ = np.sum(np.dot(Xc.T, Xc) ** 2) / n_samples ** 2
    beta = 1.0 / (n_features * n_samples) * (beta_ / n_samples - delta_)
    delta = (delta_ - 2.0 * mu * emp_cov_trace.sum() + n_features * mu ** 2) / n_features
    beta = min(beta, delta)
    shrinkage = 0 if beta == 0 else beta / delta
    emp_cov = np.dot(Xc.T, Xc) / n_samples
    shrunk = (1.0 - shrinkage) * emp_cov
    shrunk.flat[:: n_features + 1] += shrinkage * (np.trace(emp_cov) / n_features)
    return shrunk, shrinkage


ANNUALIZATION = {"daily": 252, "weekly": 52, "monthly": 12}                             # :116-124


def shrinkage_window(spec, mkt, d_idx, cols, cov_fn=None):
    """``calculate_shrinkage_portfolio`` (:703-758) in the closed form of its own CHECK block (:748-756):
    ``1/gamma * inv(Sigma_LW * f) @ (mu_hat * f)`` with f the annualisation factor.  ``cov_fn`` lets the tests plug in
    the installed ``sklearn.covariance.ledoit_wolf`` instead of the restatement above."""
    cols = np.asarray(cols)
    t, _, X = daily_statistics(spec, mkt, d_idx, cols)
    f = ANNUALIZATION[spec["rolling_window_frequency"]]
    mean = X.mean(axis=0) * f                                                           # :721-724 (compounding=False)
    cov, shrink = (cov_fn or ledoit_wolf)(X)
    cov = cov * f                                                                       # :727-729
    weights = 1 / spec["risk_aversion"] * np.dot(np.linalg.inv(cov), mean)              # :750-753
    return dict(t=t, mean=mean, cov=cov, shrinkage=shrink, weights=weights)


def clean_weights(w, cutoff=1e-4, rounding=5):
    """pypfopt 1.5.5 ``clean_weights`` (:743)."""
    w = np.array(w, dtype=np.float64, copy=True)
    w[np.abs(w) < cutoff] = 0
    return np.round(w, rounding)


def cap_order(mkt, d_idx, size, eligible=None):
    """Asset set and ORDER of one window: ``nlargest(size)`` of the caps at d (:653-654, F7)."""
    caps = mkt.caps[d_idx]
    cand = np.arange(caps.shape[0]) if eligible is None else np.asarray(eligible)
    # nlargest keeps first occurrence on ties; the generator guarantees no ties.
    order = cand[np.argsort(-caps[cand], kind="stable")]
    return order[:size]


def window_weights(spec, mkt, d_idx, cols=None, hf_lookback_days=None):
    """Dispatcher slice of ``calculate_portfolio_weights`` (:941-1052) for the in-scope strategies."""
    if cols is None:
        cols = cap_order(mkt, d_idx, spec["size"])
    strat = spec["weighting_strategy"]
    if strat.startswith("conjugate_hf_"):
        return conjugate_window(spec, mkt, d_idx, cols, hf_lookback_days)["weights"], cols
    if strat == "jeffreys":
        return jeffreys_window(spec, mkt, d_idx, cols)["weights"], cols
    if strat == "jorion":
        return jorion_window(spec, mkt, d_idx, cols)["weights"], cols
    if strat == "shrinkage":
        return clean_weights(shrinkage_window(spec, mkt, d_idx, cols)["weights"]), cols
    if strat == "vw":
        return prior_w(spec, mkt.caps[d_idx, cols]), cols
    if strat == "ew":
        return prior_w(spec, mkt.caps[d_idx, cols]), cols
    raise ValueError("Unknown weights spec.")                                           # :1050
