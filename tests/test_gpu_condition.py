"""The condition estimate of every factorised window (bp_set_condition_estimate, chol_rcond.cu).

Every route a window takes to the solver is held to the same two checks against the matrix it factorised (the S1 output
of the same call, or the caller's matrix): anorm1 within 1e-13 of its column-abs-sum max, and rcond
  * within 1e-9 of LAPACK's dpocon on np.linalg.cholesky(A) where cond_1 <= 1e6 (there the solves keep enough digits
    for dlacn2 to take the same sign and argmax decisions), and
  * inside [(1 - 100 cond_1 eps) r, 10 r], r = 1/cond_1 from a refined inverse, for every window: the estimate of
    ||A^-1||_1 is a lower bound up to the rounding of the solves.
Turning the estimate on changes no other output bit, and a window with a non-zero status gets rcond = 0 exactly.
"""
import glob
import json
import os

import numpy as np
import pandas as pd
import pytest
from scipy.linalg.lapack import dpocon

from incorporating_different_sources_b200._lib import SCAL
from incorporating_different_sources_b200.synthetic import generate_market
from incorporating_different_sources_b200.windows import ffill_rows, plan_daily_windows, plan_weekly_windows
from tests import _solver_ref as sref

pytestmark = pytest.mark.gpu

EPS = 2.0 ** -52
ANORM, RCOND = SCAL["anorm1"], SCAL["rcond"]
GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
SAME = ("weights", "nu", "w1", "status")


@pytest.fixture(scope="module")
def engine():
    from incorporating_different_sources_b200.engine import BayesEngine
    eng = BayesEngine(0)
    yield eng
    eng.set_condition_estimate(False)
    eng.close()


def _inv_norm1(A):
    """||A^-1||_1 from the float64 inverse refined once with a residual in extended precision."""
    X = np.linalg.inv(A)
    R = np.eye(A.shape[0], dtype=np.longdouble) - A.astype(np.longdouble) @ X.astype(np.longdouble)
    X = X.astype(np.longdouble) + X.astype(np.longdouble) @ R
    return float(np.max(np.sum(np.abs(X), axis=0)))


def check_windows(A, scal, status, what):
    """The two checks of the module docstring for windows A [W][N][N] (symmetric) and their scalars / status."""
    assert np.all(status == 0), f"{what}: status {status}"
    for i in range(A.shape[0]):
        a = A[i]
        anorm = float(np.max(np.abs(a).sum(axis=0)))
        assert abs(scal[i, ANORM] - anorm) <= 1e-13 * anorm, f"{what} window {i}: anorm1 {scal[i, ANORM]!r} vs {anorm!r}"
        rc = scal[i, RCOND]
        cond1 = anorm * _inv_norm1(a)
        r = 1.0 / cond1
        lo = (1.0 - 100.0 * cond1 * EPS) * r
        assert lo <= rc <= 10.0 * r, f"{what} window {i}: rcond {rc:.6e} outside [{lo:.6e}, {10 * r:.6e}] (cond_1 {cond1:.3e})"
        if cond1 <= 1e6:
            want, info = dpocon(np.asfortranarray(np.linalg.cholesky(a)), anorm, "L")
            assert info == 0
            assert abs(rc - want) <= 1e-9 * want, f"{what} window {i}: rcond {rc!r} vs dpocon {want!r}"


def _run_both(engine, fn, outputs):
    """fn(outputs) with the estimate off, then on; everything but slots 10-11 must be the same bits."""
    engine.set_condition_estimate(False)
    off = fn(outputs)
    engine.set_condition_estimate(True)
    try:
        on = fn(outputs)
    finally:
        engine.set_condition_estimate(False)
    for k in SAME:
        if k in off:
            assert np.array_equal(off[k], on[k], equal_nan=True), k
    assert np.array_equal(off["scalars"][:, :10], on["scalars"][:, :10], equal_nan=True)
    return on


def _upload(engine, mkt, hf=True):
    engine.upload_market(prices=mkt.prices, caps=mkt.caps, hf_prices=mkt.hf_prices if hf else None,
                         mcm=np.stack([mkt.vix, mkt.epu]), rf_row=ffill_rows(mkt.dates, mkt.dates, mkt.rf))


# --------------------------------------------------------------------------------- 1. conjugate and Jeffreys batches
@pytest.mark.parametrize("N", [10, 33, 64, 90, 500])
def test_conjugate_and_jeffreys(engine, N):
    rw = 2 * N + 40                 # n - 1 > N: the Jeffreys windows are full rank
    n_days = rw + 8
    mkt = generate_market(N, n_days, seed=500 + N)
    _upload(engine, mkt)
    d_idx = list(range(n_days - 4, n_days))
    spec = dict(weighting_strategy="conjugate_hf_vix_vw", size=N, risk_aversion=5, rolling_window=rw,
                rolling_window_frequency="daily", mcm_scaling=1)
    cb = plan_daily_windows(spec, mkt.dates, d_idx, mkt.hf_ts, hf_lookback_days=7)
    outs = ("weights", "nu", "w1", "status", "scalars", "S1")
    got = _run_both(engine, lambda o: engine.conjugate(cb, outputs=o), outs)
    check_windows(got["S1"], got["scalars"], got["status"], f"conjugate N={N}")
    jb = plan_daily_windows(dict(spec, weighting_strategy="jeffreys"), mkt.dates, d_idx, need_hf=False)
    got = _run_both(engine, lambda o: engine.jeffreys(jb, outputs=o), outs)
    check_windows(got["S1"], got["scalars"], got["status"], f"jeffreys N={N}")


# --------------------------------------------------------------------------------- 2. every route
@pytest.fixture(scope="module")
def wave_market():
    return generate_market(33, 620, seed=77)


def test_full_wave_and_chunked_workspace(engine, wave_market):
    """560 windows: more than the cluster kernel takes (chol_solve_kernel), then the same batch in workspace chunks
    of about 80 windows."""
    mkt = wave_market
    _upload(engine, mkt)
    spec = dict(weighting_strategy="conjugate_hf_vix_vw", size=33, risk_aversion=5, rolling_window=60,
                rolling_window_frequency="daily", mcm_scaling=1)
    cb = plan_daily_windows(spec, mkt.dates, list(range(60, 620)), mkt.hf_ts, hf_lookback_days=7)
    outs = ("weights", "nu", "w1", "status", "scalars", "S1")
    full = _run_both(engine, lambda o: engine.conjugate(cb, outputs=o), outs)
    check_windows(full["S1"], full["scalars"], full["status"], "full wave")
    per = (33 + 31) // 32 * 32
    engine.set_workspace_limit(50 * 8 * ((per + 8) * per + 9 * 48 + 12 + 4096))
    try:
        chunked = _run_both(engine, lambda o: engine.conjugate(cb, outputs=o), outs)
    finally:
        engine.set_workspace_limit(24 << 30)
    np.testing.assert_allclose(chunked["scalars"][:, RCOND], full["scalars"][:, RCOND], rtol=1e-12, atol=0)
    np.testing.assert_allclose(chunked["scalars"][:, ANORM], full["scalars"][:, ANORM], rtol=1e-13, atol=0)


def test_pipelined_upload(engine):
    import torch
    mkt = generate_market(40, 1100, seed=23)
    spec = dict(weighting_strategy="conjugate_hf_vix_vw", size=40, risk_aversion=5, rolling_window=60,
                rolling_window_frequency="daily", mcm_scaling=1)
    batch = plan_daily_windows(spec, mkt.dates, list(range(60, 1100)), mkt.hf_ts, hf_lookback_days=7)
    arrays = dict(prices=mkt.prices, caps=mkt.caps, hf_prices=mkt.hf_prices, mcm=np.stack([mkt.vix, mkt.epu]),
                  rf_row=ffill_rows(mkt.dates, mkt.dates, mkt.rf))
    outs = ("weights", "nu", "w1", "status", "scalars")
    engine.set_condition_estimate(True)
    try:
        engine.upload_market(**arrays)
        ref = engine.conjugate(batch, outputs=outs + ("S1",))
        pinned = {k: torch.from_numpy(np.ascontiguousarray(v)).pin_memory() for k, v in arrays.items()}
        engine.set_upload_pipeline(8, 0)
        engine.upload_market(**{k: v.numpy() for k, v in pinned.items()}, async_copy=True)
        got = engine.conjugate(batch, outputs=outs)
        engine.synchronize()
    finally:
        engine.set_upload_pipeline()
        engine.set_condition_estimate(False)
    for k in outs:
        assert np.array_equal(got[k], ref[k]), k
    # the S1 of the blocking call: the pipelined call solves the early windows before the matrices could be read back
    check_windows(ref["S1"][::13], got["scalars"][::13], got["status"][::13], "pipelined")


@pytest.mark.parametrize("which", ["jorion", "shrinkage"])
def test_estimators(engine, which):
    N = 40
    mkt = generate_market(N, 200, seed=91)
    _upload(engine, mkt, hf=False)
    spec = dict(weighting_strategy=which, size=N, risk_aversion=5, rolling_window=120, rolling_window_frequency="daily",
                mcm_scaling=None)
    b = plan_daily_windows(spec, mkt.dates, list(range(190, 200)), need_hf=False)
    run = getattr(engine, which)
    got = _run_both(engine, lambda o: run(b, outputs=o), ("weights", "nu", "w1", "status", "scalars", "S1"))
    check_windows(got["S1"], got["scalars"], got["status"], which)


def test_weekly_windows(engine):
    n = 20
    mkt = generate_market(n, 460, seed=1234)
    _upload(engine, mkt)
    spec = dict(weighting_strategy="conjugate_hf_epu_vw", size=n, risk_aversion=5, rolling_window=70,
                rolling_window_frequency="weekly", mcm_scaling=2)
    rows, cb = plan_weekly_windows(spec, mkt.dates, list(range(450, 460)), mkt.dates, mkt.rf,
                                   np.stack([mkt.vix, mkt.epu]), mkt.hf_ts)
    engine.set_resampled(rows)
    got = _run_both(engine, lambda o: engine.conjugate(cb, outputs=o), ("weights", "nu", "w1", "status", "scalars", "S1"))
    check_windows(got["S1"], got["scalars"], got["status"], "weekly conjugate")
    _, jb = plan_weekly_windows(dict(spec, weighting_strategy="jeffreys"), mkt.dates, list(range(450, 460)), mkt.dates,
                                mkt.rf, None, need_hf=False)
    got = _run_both(engine, lambda o: engine.jeffreys(jb, outputs=o), ("weights", "nu", "w1", "status", "scalars", "S1"))
    check_windows(got["S1"], got["scalars"], got["status"], "weekly jeffreys")


@pytest.mark.parametrize("N", [1, 2, 31, 64, 257])
def test_caller_matrices(engine, N):
    """engine.solve on matrices with cond from 1e2 to ~1e12 (the last: positive pivots, the case the pivot check
    misses), one and two right-hand sides."""
    rng = np.random.default_rng(700 + N)
    kappas = [1e2, 1e4, 1e6, 1e9, 1e12] if N > 1 else [1.0]
    S = np.stack([sref.spd_with_kappa(N, k, rng) if N > 1 else np.array([[3.5]]) for k in kappas])
    rhs = rng.standard_normal((len(kappas), N))
    got = _run_both(engine, lambda o: engine.solve(S, rhs, jeffreys=True, outputs=o), ("weights", "nu", "w1", "status", "scalars"))
    check_windows(S, got["scalars"], got["status"], f"solve N={N}")
    if N == 1:
        assert got["scalars"][0, RCOND] == pytest.approx(1.0, rel=1e-15)        # 1 / (|A^-1| anorm1)
    if N >= 31:
        engine.set_condition_estimate(True)
        try:
            j = engine.solve(S, rhs, jorion=True, n_returns=N + 40)
        finally:
            engine.set_condition_estimate(False)
        check_windows(S, j["scalars"], j["status"], f"solve jorion N={N}")


def test_dense_posterior(engine):
    rng = np.random.default_rng(5)
    N = 45
    X = rng.standard_normal((120, N))
    T, t = X.T @ X, X.sum(axis=0)
    engine.set_condition_estimate(True)
    try:
        res = engine.dense_posterior(jeffreys=True, rolling_window=121, risk_aversion=5.0, T=T, t=t)
    finally:
        engine.set_condition_estimate(False)
    check_windows(res["S1"][None], res["scalars"][None], res["status"], "dense_posterior")


# --------------------------------------------------------------------------------- 3. failures
def test_indefinite_caller_matrix(engine):
    rng = np.random.default_rng(9)
    N = 50
    good = sref.spd_with_kappa(N, 1e3, rng)
    bad = good.copy()
    bad[30, 30] = -1.0
    engine.set_condition_estimate(True)
    try:
        res = engine.solve(np.stack([good, bad, good]), rng.standard_normal((3, N)))
    finally:
        engine.set_condition_estimate(False)
    assert res["status"][1] != 0 and res["scalars"][1, RCOND] == 0.0
    check_windows(np.stack([good, good]), res["scalars"][[0, 2]], res["status"][[0, 2]], "neighbours of a failure")


def test_conjugate_window_without_returns(engine):
    """Every bar of one stock missing on the trade date: with a one-day look-back the window keeps no intraday return,
    S1 is NaN, the status is non-zero and rcond is 0."""
    N = 12
    mkt = generate_market(N, 80, seed=31)
    bars = len(mkt.hf_ts) // mkt.n_days
    hf = mkt.hf_prices.copy()
    hf[75 * bars:76 * bars, 3] = np.nan
    engine.upload_market(prices=mkt.prices, caps=mkt.caps, hf_prices=hf, mcm=np.stack([mkt.vix, mkt.epu]),
                         rf_row=ffill_rows(mkt.dates, mkt.dates, mkt.rf))
    spec = dict(weighting_strategy="conjugate_hf_vix_vw", size=N, risk_aversion=5, rolling_window=40,
                rolling_window_frequency="daily", mcm_scaling=1)
    cb = plan_daily_windows(spec, mkt.dates, [74, 75, 76], mkt.hf_ts, hf_lookback_days=1)
    engine.set_condition_estimate(True)
    try:
        res = engine.conjugate(cb, outputs=("status", "scalars"))
    finally:
        engine.set_condition_estimate(False)
    assert res["scalars"][1, SCAL["m"]] < 2 and res["status"][1] != 0
    assert res["scalars"][1, RCOND] == 0.0
    assert np.all(res["status"][[0, 2]] == 0) and np.all(res["scalars"][[0, 2], RCOND] > 0)


def test_jeffreys_rank_deficient(engine):
    """n - 1 < N returns (SURVEY F6): a failed pivot or an rcond that says so, never status 0 with a healthy rcond."""
    N = 40
    mkt = generate_market(N, 120, seed=41)
    _upload(engine, mkt, hf=False)
    spec = dict(weighting_strategy="jeffreys", size=N, risk_aversion=5, rolling_window=30, rolling_window_frequency="daily")
    jb = plan_daily_windows(spec, mkt.dates, list(range(100, 120)), need_hf=False)
    engine.set_condition_estimate(True)
    try:
        res = engine.jeffreys(jb, outputs=("status", "scalars"))
    finally:
        engine.set_condition_estimate(False)
    for i in range(20):
        assert res["status"][i] != 0 or res["scalars"][i, RCOND] < 1e-12, (i, res["scalars"][i, RCOND])
        if res["status"][i] != 0:
            assert res["scalars"][i, RCOND] == 0.0


# --------------------------------------------------------------------------------- 4. nothing else moves
def test_jeffreys_chain_is_skipped(engine):
    N = 33
    mkt = generate_market(N, 200, seed=57)
    _upload(engine, mkt, hf=False)
    spec = dict(weighting_strategy="jeffreys", size=N, risk_aversion=5, rolling_window=120, rolling_window_frequency="daily")
    jb = plan_daily_windows(spec, mkt.dates, list(range(140, 200)), need_hf=False)
    outs = ("weights", "nu", "w1", "status", "scalars")
    engine.solve_work()
    engine.jeffreys(jb, outputs=outs)
    assert engine.solve_work()["chained"] > 0                 # the chain is used with the estimate off
    engine.set_jeffreys_chain(0)
    try:
        per_window = engine.jeffreys(jb, outputs=outs)
    finally:
        engine.set_jeffreys_chain(8)
    engine.solve_work()
    engine.set_condition_estimate(True)
    try:
        on = engine.jeffreys(jb, outputs=outs)
        work = engine.solve_work()
    finally:
        engine.set_condition_estimate(False)
    assert work["chained"] == 0 and work["factored"] == 60
    for k in SAME:
        assert np.array_equal(on[k], per_window[k]), k
    assert np.array_equal(on["scalars"][:, :10], per_window["scalars"][:, :10])
    assert np.all(on["scalars"][:, RCOND] > 0)


def test_stage_timing(engine):
    rng = np.random.default_rng(1)
    S = np.stack([sref.spd_with_kappa(64, 1e3, rng) for _ in range(4)])
    engine.set_stage_timing(True)
    engine.stage_times()
    engine.set_condition_estimate(True)
    try:
        engine.solve(S, rng.standard_normal((4, 64)))
    finally:
        engine.set_condition_estimate(False)
    st = engine.stage_times()
    engine.solve(S, rng.standard_normal((4, 64)))
    st_off = engine.stage_times()
    engine.set_stage_timing(False)
    assert st["cond"]["launches"] == 2 and st["cond"]["ms"] > 0
    assert st_off["cond"]["launches"] == 0


# --------------------------------------------------------------------------------- 5. backtest_portfolio
def _golden_backtest(name, **kw):
    from incorporating_different_sources_b200 import portfolio_calculations as pc
    z = np.load(os.path.join(GOLD, name + ".npz"))
    meta = json.loads(str(z["meta"]))
    mkt = generate_market(**meta["market"])
    md = mkt.market_data()
    if meta.get("damage"):
        from tests.golden.make_backtest_golden import apply_damage
        md = apply_damage(md, meta["damage"])
    return meta, mkt, pc.backtest_portfolio(meta["spec"], pd.Timestamp(meta["start"]), pd.Timestamp(meta["end"]), md, **kw)


GOLDEN_BT = sorted(os.path.basename(p)[:-4] for p in glob.glob(os.path.join(GOLD, "bt_*.npz")))


@pytest.mark.parametrize("name", GOLDEN_BT)
def test_backtest_keywords_none_change_nothing(name):
    meta, _, a = _golden_backtest(name)
    _, _, b = _golden_backtest(name, min_rcond=None, diagnostics=None)
    assert set(a) == set(b)
    for k in a:
        assert a[k].equals(b[k]), k
    diag = {}
    _, _, c = _golden_backtest(name, diagnostics=diag)
    for k in a:
        assert a[k].equals(c[k]), k
    rc = diag["rcond"]
    assert rc.name == meta["spec"]["display_name"]
    assert list(rc.index) == list(a["portfolio_weights_metrics_df"].index)
    if meta["spec"]["weighting_strategy"] in ("vw", "ew"):
        assert rc.isna().all()
    else:
        assert (rc > 0).all() and np.isfinite(rc).all()


def test_backtest_diagnostics_and_threshold():
    from incorporating_different_sources_b200 import portfolio_calculations as pc
    from incorporating_different_sources_b200.engine import upload_synthetic
    name = "bt_jeffreys_monthly_n6"
    diag = {}
    meta, mkt, _ = _golden_backtest(name, diagnostics=diag)
    rc = diag["rcond"]
    assert rc.name == meta["spec"]["display_name"]
    eng = pc._engine()
    assert not eng.condition_estimate                         # restored after the backtest
    upload_synthetic(eng, mkt)
    d_idx = [int(np.searchsorted(mkt.dates, np.datetime64(d))) for d in rc.index.values]
    jb = plan_daily_windows(meta["spec"], mkt.dates, d_idx, need_hf=False)
    eng.set_condition_estimate(True)
    try:
        res = eng.jeffreys(jb, outputs=("scalars", "status"))
    finally:
        eng.set_condition_estimate(False)
    np.testing.assert_allclose(rc.to_numpy(), res["scalars"][:, RCOND], rtol=1e-12, atol=0)
    k = int(np.argmin(rc.to_numpy()))
    with pytest.raises(np.linalg.LinAlgError, match=str(rc.index[k].date())):
        _golden_backtest(name, min_rcond=float(rc.iloc[k]) * (1 + 1e-9))
    assert not eng.condition_estimate
    _golden_backtest(name, min_rcond=float(rc.iloc[k]) * (1 - 1e-9))
