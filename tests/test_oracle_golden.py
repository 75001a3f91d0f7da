"""The NumPy oracle (oracle/bayes_oracle.py) against the reference's own outputs.

The golden vectors were produced by the unmodified reference (tests/golden/make_golden.py);
this pins the oracle.  Tolerance 1e-12 relative (only summation order may differ);
index order is compared exactly.
"""
import numpy as np
import pytest

from oracle import bayes_oracle as bo
from tests._golden import check_matrix, estimator_golden_names, golden_names, load_golden, market_for, relerr

TOL = 1e-12


@pytest.mark.parametrize("name", golden_names())
def test_oracle_matches_reference(name):
    z, meta = load_golden(name)
    mkt = market_for(meta)
    spec = meta["spec"]
    for wi, w in enumerate(meta["windows"]):
        pre = f"w{wi}_"
        d_idx = w["d_idx"]
        cols = bo.cap_order(mkt, d_idx, spec["size"])
        assert np.array_equal(cols, z[pre + "cols"]), "asset set / cap-descending order must be bit-exact"
        if spec["weighting_strategy"].startswith("conjugate"):
            r = bo.conjugate_window(spec, mkt, d_idx, cols, hf_lookback_days=meta["hf_days"])
            for k in ("n0", "n1", "c", "v1"):
                assert abs(r[k] - float(z[pre + k])) <= TOL * abs(float(z[pre + k])), k
            for k in ("t", "w0"):
                assert relerr(r[k], z[pre + k]) <= TOL, k
            for k in ("T", "S0", "S1"):
                check_matrix(k, r[k], z, pre, TOL)
            # the solve is conditioned by cond(S1): allow cond * eps on the solved quantities
            tol_solve = max(TOL, 50 * float(z[pre + "cond_S1"]) * np.finfo(float).eps)
            for k in ("w1", "nu", "weights"):
                assert relerr(r[k], z[pre + k]) <= tol_solve, k
        else:
            r = bo.jeffreys_window(spec, mkt, d_idx, cols)
            assert relerr(r["t"], z[pre + "t"]) <= TOL
            check_matrix("T", r["T"], z, pre, TOL)
            tol_solve = max(TOL, 50 * float(z[pre + "cond_J"]) * np.finfo(float).eps)
            for k in ("nu", "weights"):
                assert relerr(r[k], z[pre + k]) <= tol_solve, k


@pytest.mark.parametrize("name", estimator_golden_names())
def test_estimator_oracles_match_reference(name):
    """Jorion against the unmodified reference's ``calculate_jorion_portfolio``; the shrinkage closed form (and the
    NumPy restatement of sklearn's ``ledoit_wolf``) against sklearn on the reference's own excess returns."""
    z, meta = load_golden(name)
    mkt = market_for(meta)
    spec = meta["spec"]
    eps = np.finfo(float).eps
    for wi, w in enumerate(meta["windows"]):
        pre = f"w{wi}_"
        d_idx = w["d_idx"]
        cols = bo.cap_order(mkt, d_idx, spec["size"])
        assert np.array_equal(cols, z[pre + "cols"]), "asset set / cap-descending order must be bit-exact"
        r = bo.jorion_window(spec, mkt, d_idx, cols)
        tol = max(TOL, 50 * float(z[pre + "cond_V"]) * eps)
        assert relerr(r["weights"], z[pre + "jorion_weights"]) <= tol
        for k, g in (("mu_g", "jorion_mu_g"), ("lambda_hat", "jorion_lambda"), ("v_hat", "jorion_v")):
            assert abs(r[k] - float(z[pre + g])) <= tol * abs(float(z[pre + g])), k
        s = bo.shrinkage_window(spec, mkt, d_idx, cols)
        tol = max(TOL, 50 * float(z[pre + "cond_LW"]) * eps)
        assert abs(s["shrinkage"] - float(z[pre + "lw_shrinkage"])) <= 1e-10 * float(z[pre + "lw_shrinkage"])
        assert relerr(np.diag(s["cov"]), z[pre + "lw_cov_diag"]) <= TOL
        assert relerr(s["cov"][0], z[pre + "lw_cov_row0"]) <= TOL
        assert relerr(s["weights"], z[pre + "lw_weights"]) <= tol


def test_ledoit_wolf_restatement_matches_installed_sklearn():
    """pypfopt's CovarianceShrinkage.ledoit_wolf() is sklearn.covariance.ledoit_wolf: pin the restatement on it."""
    sk = pytest.importorskip("sklearn.covariance")
    rng = np.random.default_rng(11)
    for m, n in ((251, 10), (59, 25), (400, 130), (30, 40)):
        X = rng.standard_normal((m, n)) @ np.diag(rng.uniform(0.005, 0.03, n)) + 4e-4
        X[:, : n // 2] += 0.01 * rng.standard_normal((m, 1))          # a common factor
        cov, sh = sk.ledoit_wolf(X)
        cov2, sh2 = bo.ledoit_wolf(X)
        assert abs(sh - sh2) <= 1e-12 * max(abs(sh), 1e-300)
        assert relerr(cov2, cov) <= 1e-13


def test_ledoit_wolf_one_feature_has_zero_shrinkage_as_in_sklearn():
    """sklearn returns shrinkage 0 and the plain variance for one feature, whatever its beta and delta round to (the
    general formula's delta is 0 in exact arithmetic there, and rounding leaves it of either sign)."""
    sk = pytest.importorskip("sklearn.covariance")
    rng = np.random.default_rng(12)
    for m in (2, 3, 17, 120, 251):
        for _ in range(20):
            X = rng.standard_normal((m, 1)) * rng.uniform(0.005, 0.03) + 4e-4
            cov, sh = sk.ledoit_wolf(X)
            cov2, sh2 = bo.ledoit_wolf(X)
            assert sh == 0.0 and sh2 == 0.0
            assert cov2.shape == (1, 1) and relerr(cov2, cov) <= 1e-15


def test_weekly_resample_matches_pandas():
    import pandas as pd
    from incorporating_different_sources_b200.synthetic import generate_market
    mkt = generate_market(3, 90, seed=5)
    df = pd.DataFrame(mkt.prices, index=pd.DatetimeIndex(mkt.dates))
    for end in (40, 61, 89):
        ref = df.iloc[: end + 1].resample("W").last()
        lab, val, _ = bo.resample_weekly_last(mkt.dates[: end + 1], mkt.prices[: end + 1])
        assert np.array_equal(ref.index.values.astype("datetime64[ns]"), lab)
        assert np.array_equal(ref.values, val)
