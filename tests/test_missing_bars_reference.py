"""The intraday prior with missing bars, on the CPU: the dropna restatement the GPU tests compare against
(tests/_dropna_ref.py) is pinned to the reference's own pandas expression (portfolio_calculations.py:314-318),
and the rule the CUDA path is built on -- one keep mask per working market serves every window -- is checked."""
import numpy as np
import pandas as pd
import pytest

from oracle import bayes_oracle as bo
from oracle.ref_import import load_reference, reference_available
from tests._dropna_ref import keep_mask, realized_covariance_dropna

needs_reference = pytest.mark.skipif(not reference_available(), reason="reference sources not present on this machine")
BARS = 26


def _pandas_prior(P):
    """The reference's expression, verbatim (:314, :317-318)."""
    df = pd.DataFrame(P)
    h = np.log(df / df.shift(1)).dropna()
    return (h.cov() * len(h)).to_numpy(), len(h)


def _prices(n_rows, n_cols, seed):
    rng = np.random.default_rng(seed)
    return 50.0 * np.exp(np.cumsum(0.002 * rng.standard_normal((n_rows, n_cols)), axis=0))


def _holes(kind, P):
    P = P.copy()
    if kind == "isolated":
        P[[5, 17, 40], [0, 3, 1]] = np.nan
    elif kind == "adjacent":
        P[[10, 11, 12], 2] = np.nan
        P[13, 4] = np.nan
    elif kind == "first_and_last":
        P[0, 1] = np.nan
        P[-1, 3] = np.nan
    elif kind == "whole_day":
        P[2 * BARS:3 * BARS, 5] = np.nan
    elif kind == "m1":
        P[:-2, 0] = np.nan                  # only the last two bars are complete: one return
    elif kind == "m0":
        P[::2, 1] = np.nan                  # every return touches a hole
    return P


@pytest.mark.parametrize("kind,expect_m", [("isolated", None), ("adjacent", None), ("first_and_last", None),
                                           ("whole_day", None), ("m1", 1), ("m0", 0)])
def test_dropna_prior_matches_pandas(kind, expect_m):
    P = _holes(kind, _prices(5 * BARS, 6, seed=11))
    got, m = realized_covariance_dropna(P)
    ref, m_ref = _pandas_prior(P)
    assert m == m_ref
    if expect_m is not None:
        assert m == expect_m and np.isnan(got).all() and np.isnan(ref).all()
        return
    assert m < P.shape[0] - 1
    assert np.allclose(got, ref, rtol=1e-12, atol=0)


def test_dropna_prior_counts_two_returns_per_hole():
    P = _prices(60, 4, seed=3)
    P[30, 2] = np.nan                       # one bar: returns 30 and 31 go, nothing bridges the gap
    _, m = realized_covariance_dropna(P)
    assert m == 59 - 2
    P[0, 0] = np.nan                        # the first bar: return 1 goes
    _, m = realized_covariance_dropna(P)
    assert m == 59 - 3


@pytest.mark.parametrize("seed", [0, 1, 2])
def test_dropna_prior_is_the_oracle_on_clean_windows(seed):
    P = _prices(3 * BARS + seed, 7, seed=seed)
    got, m = realized_covariance_dropna(P)
    ref, m_ref = bo.realized_covariance(P)
    assert m == m_ref and np.array_equal(got, ref)


def test_one_keep_mask_per_market_serves_every_window():
    """Return row r needs price rows r-1 and r only, both inside any window [lo, hi) with lo < r < hi, so the rows a
    window's own dropna keeps are exactly the market mask's rows inside (lo, hi)."""
    rng = np.random.default_rng(7)
    R, N = 40 * BARS, 9
    P = _prices(R, N, seed=8)
    P[rng.integers(0, R, 120), rng.integers(0, N, 120)] = np.nan          # isolated holes
    P[5 * BARS:6 * BARS, 4] = np.nan                                      # a stock missing a whole day
    P[rng.integers(0, R, 10)] = np.nan                                    # whole rows
    keep = keep_mask(P)
    for _ in range(300):
        lo = int(rng.integers(0, R - 3))
        hi = int(rng.integers(lo + 3, min(R, lo + 8 * BARS) + 1))
        df = pd.DataFrame(P[lo:hi])
        kept = np.log(df / df.shift(1)).dropna().index.to_numpy() + lo
        assert np.array_equal(kept, lo + 1 + np.nonzero(keep[lo + 1:hi])[0])
        _, m = realized_covariance_dropna(P[lo:hi])
        assert m == keep[lo + 1:hi].sum()


@needs_reference
@pytest.mark.parametrize("kind", ["isolated", "whole_day", "m0"])
def test_dropna_prior_matches_reference_function(kind):
    """``calculate_conjugate_prior_S`` of the reference itself on an intraday frame with missing bars."""
    from incorporating_different_sources_b200.synthetic import generate_market
    ref = load_reference()
    mkt = generate_market(6, 40, seed=5, bars_per_day=BARS)
    spec = dict(weighting_strategy="conjugate_hf_vix_vw", size=6, risk_aversion=5, rolling_window=20,
                rolling_window_frequency="weekly", mcm_scaling=1)
    d_idx = 35
    d = pd.Timestamp(mkt.dates[d_idx])
    lo, hi = bo.hf_window_rows(spec, mkt.hf_ts, mkt.dates[d_idx])
    H = mkt.hf_prices.copy()
    H[lo:hi] = _holes(kind, H[lo:hi])
    md = mkt.market_data()
    intr = pd.DataFrame(H, index=md["stock_intraday_prices_df"].index, columns=md["stock_intraday_prices_df"].columns)
    intr = intr.loc[intr.index <= d.replace(hour=23, minute=59, second=59)]
    n0 = 123.0
    got = ref.calculate_conjugate_prior_S(spec, d, intr, md["vix_prices_df"].loc[:d], conjugate_prior_n=n0)
    want, m = realized_covariance_dropna(H[lo:hi])
    if m < 2:
        assert np.isnan(got.to_numpy()).all()
    else:
        assert np.allclose(got.to_numpy(), n0 * want, rtol=1e-12, atol=0)
