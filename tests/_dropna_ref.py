"""NumPy restatement of the reference's intraday prior with missing bars (portfolio_calculations.py:314-318):

    h = np.log(df / df.shift(1)).dropna();  S0 = n0 * h.cov() * len(h)

``realized_covariance_dropna`` is ``oracle.bayes_oracle.realized_covariance`` with the return rows that hold a
NaN in any column dropped first; on NaN-free windows it is the same computation on the same array.
``use_dropna_oracle`` makes the oracle's window functions use it (for tests that punch holes into a market).
"""
import numpy as np


def realized_covariance_dropna(hf_prices_window):
    h = np.log(hf_prices_window[1:] / hf_prices_window[:-1])
    h = h[~np.isnan(h).any(axis=1)]
    m = h.shape[0]
    if m < 2:                                           # pandas' cov of < 2 rows is all NaN
        n = hf_prices_window.shape[1]
        return np.full((n, n), np.nan), m
    return np.cov(h.T) * m, m


def keep_mask(hf_prices):
    """Per working market: return row r (log of price row r over row r-1) is kept iff none of its returns is NaN."""
    keep = np.zeros(hf_prices.shape[0], dtype=bool)
    with np.errstate(invalid="ignore", divide="ignore"):
        keep[1:] = ~np.isnan(np.log(hf_prices[1:] / hf_prices[:-1])).any(axis=1)
    return keep


def use_dropna_oracle(monkeypatch):
    from oracle import bayes_oracle as bo
    monkeypatch.setattr(bo, "realized_covariance", realized_covariance_dropna)
