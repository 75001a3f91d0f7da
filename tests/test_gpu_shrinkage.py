"""The Ledoit-Wolf shrinkage stage (estimators.cu lw_shrink_kernel) on its own: every window's scalars (shrinkage, mu,
beta, delta), S1 diagonal, rhs, weights, nu, w1 and status against the extended-precision reference of
tests/_lw_ref.py and its a-priori bounds, at the kernel's column and row edges, for N >= m, clipped (s = 1) and
near-clipped windows, one asset, weekly windows, a chunked batch and both Gram routes.  Each case asserts its route
from the work counters; the planner never chains shrinkage.  Where Jorion runs on the same batch, the S1 off-diagonal
is Jorion's S1 bit for bit (the stage rewrites only the diagonal)."""
import numpy as np
import pandas as pd
import pytest

from oracle import bayes_oracle as bo
from tests import _gram_ref as gr
from tests import _lw_ref as lr

pytestmark = pytest.mark.gpu

U = lr.U
LD = np.longdouble
GAMMA = 3.0
NO_REUSE = 2 ** 31 - 1
OUTS = ("weights", "nu", "w1", "rhs", "scalars", "status", "S1")
SC = dict(shrinkage=0, mu=1, beta=2, delta=4, anorm1=10, rcond=11)
WORST = {}                 # case -> output -> worst |E| / bound (printed at the end of the module)


@pytest.fixture(scope="module")
def engine():
    from incorporating_different_sources_b200.engine import BayesEngine
    gr.require_extended_precision()
    eng = BayesEngine(0)
    yield eng
    eng.close()
    if WORST:
        print("\nworst |E| / bound per case:")
        for case, d in WORST.items():
            print(f"  {case:34s} " + " ".join(f"{k}={v:.3g}" for k, v in sorted(d.items())))


def _assert_ratio(case, name, r, i):
    d = WORST.setdefault(case, {})
    d[name] = max(d.get(name, 0.0), r)
    assert r < 1.0, f"{case}: {name} of window {i} is {r:.3g} x its bound"


def _spec(N, n, freq="daily", strategy="shrinkage"):
    return dict(weighting_strategy=strategy, size=N, risk_aversion=GAMMA, turnover_cost=15,
                rebalancing_frequency="daily", rolling_window=n, rolling_window_frequency=freq, mcm_scaling=None,
                display_name="x")


def _market(N, D, seed, iid=False, rf_mode="varying"):
    """A seeded factor-model market, or with ``iid`` i.i.d. equal-volatility log returns (where the intensity clips)."""
    from incorporating_different_sources_b200.synthetic import generate_market
    mkt = generate_market(N, D, seed=seed, bars_per_day=2, rf_mode=rf_mode)
    if iid:
        R = lr.iid_returns(D, N, np.random.default_rng(seed))
        _set_log_returns(mkt, R)
    return mkt


def _set_log_returns(mkt, R):
    """Daily prices with log returns R (row 0 is the first price's row; its return is ignored)."""
    P = 100.0 * np.exp(np.cumsum(R, axis=0))
    mkt.prices[:] = P
    mkt.caps[:] = P * np.arange(1, P.shape[1] + 1)[::-1]
    mkt.hf_prices[:] = np.repeat(P, len(mkt.hf_ts) // len(mkt.dates), axis=0)


def _upload(engine, mkt):
    from incorporating_different_sources_b200.engine import upload_synthetic
    upload_synthetic(engine, mkt)


def _plan(mkt, n, d_idx):
    from incorporating_different_sources_b200.windows import plan_daily_windows
    return plan_daily_windows(_spec(mkt.n_assets, n), mkt.dates, list(d_idx), need_hf=False)


def _rf_row(mkt):
    from incorporating_different_sources_b200.windows import ffill_rows
    return ffill_rows(mkt.dates, mkt.dates, mkt.rf)


def _daily_rows(engine, mkt, batch, i):
    """(X, a, x_err) of daily window i: the device's own excess returns, which the kernel re-forms bit for bit."""
    from incorporating_different_sources_b200.windows import slice_batch
    X = engine.excess_returns(slice_batch(batch, i, i + 1))
    a = gr.daily_adjustments(_rf_row(mkt), gr.daily_return_rows(int(batch.day_row[i]), batch.rolling_window),
                             int(batch.span_days[i]))
    return X, a, 0.0


def run(case, engine, batch, *, consecutive=False, cond=False):
    """The batch with every output, its route asserted from the work counters: every window factorised, none chained.
    A consecutive batch of 16 or more windows also runs without S1 (the only output that keeps Jeffreys batches off
    the chain) and must neither chain nor change a bit of its weights."""
    W = batch.n_windows
    engine.solve_work()
    engine.gram_work()
    got = engine.shrinkage(batch, outputs=OUTS)
    sw, gw = engine.solve_work(), engine.gram_work()
    assert sw == {"factored": W, "chained": 0}, (case, sw)
    if consecutive:
        assert W >= 16 and np.all(np.diff(batch.day_row) == 1)
        assert engine.jeffreys_chain >= 2 and not cond
        lean = engine.shrinkage(batch, outputs=("weights", "nu", "status"))
        sw2 = engine.solve_work()
        assert sw2 == {"factored": W, "chained": 0}, (case, sw2)
        assert np.array_equal(lean["weights"], got["weights"]) and np.array_equal(lean["nu"], got["nu"])
    return got, gw


def check(case, engine, mkt, batch, got, windows, rows=None, jorion=None, sklearn=False):
    """Hold the listed windows to the bounds.  ``rows(i)`` -> (X, a, x_err) (default: the device's daily rows);
    ``jorion``: Jorion's S1 of the same batch and Gram route; ``sklearn``: also compare the weights with sklearn's.
    The stage's input C is the S1 off-diagonal, which only a clipped window rewrites (to zero): there the input is
    Jorion's S1, which equals the S1 of every other window bit for bit."""
    rows = rows or (lambda i: _daily_rows(engine, mkt, batch, i))
    refs = {}
    for i in windows:
        X, a, x_err = rows(i)
        S1 = got["S1"][i]
        assert np.array_equal(S1, S1.T), (case, i)
        clipped = got["scalars"][i][SC["shrinkage"]] == 1.0
        if clipped and jorion is None and X.shape[1] > 1:
            pytest.fail(f"{case}: window {i} clipped, and no Jorion S1 holds the stage's input C")
        ref = lr.LWRef(X, jorion[i] if clipped else S1, a, x_err)
        refs[i] = ref
        sc = got["scalars"][i]
        s_k, mu_k = float(sc[SC["shrinkage"]]), float(sc[SC["mu"]])
        _assert_ratio(case, "shrinkage", lr.ratio(s_k, ref.s, ref.e_s), i)
        _assert_ratio(case, "mu", lr.ratio(mu_k, ref.mu, ref.e_mu), i)
        _assert_ratio(case, "beta", lr.ratio(sc[SC["beta"]], ref.beta, ref.e_beta), i)
        _assert_ratio(case, "delta", lr.ratio(sc[SC["delta"]], ref.delta, ref.e_delta), i)
        if ref.N == 1:
            assert s_k == 0.0, (case, i, s_k)
        d, d_err = ref.diag_expected(s_k, mu_k)
        _assert_ratio(case, "S1 diag", lr.ratio(np.diag(S1), d, d_err), i)
        if s_k == 1.0:
            assert not np.any(np.tril(S1, -1)), (case, i)
            assert np.all(np.diag(S1) == np.float64(mu_k) * np.float64(ref.m)), (case, i)
        rhs, rhs_err = ref.rhs_expected(s_k)
        _assert_ratio(case, "rhs", lr.ratio(got["rhs"][i], rhs, rhs_err), i)
        if jorion is not None and s_k != 1.0:
            assert np.array_equal(np.tril(jorion[i], -1), np.tril(S1, -1)), (case, i)
        x, eps = ref.solution()
        if x is None:                       # m = 2: C has rank 1 and s is 0 in exact arithmetic (see _lw_ref)
            continue
        assert got["status"][i] == 0, (case, i, got["status"][i])
        xf = x.astype(np.float64)
        scale = float(np.max(np.abs(xf)))
        for k in ("nu", "w1"):
            _assert_ratio(case, k, float(np.max(np.abs(got[k][i] - xf))) / (eps * scale), i)
        _assert_ratio(case, "weights", float(np.max(np.abs(got["weights"][i] - xf / GAMMA)))
                      / ((eps + 2 * U) * scale / GAMMA), i)
        if sklearn:
            w_sk, s_sk = lr.sklearn_weights(X, GAMMA)
            assert abs(s_sk - float(ref.s)) <= lr.LWRef(X, ref.C_off, a, x_err, lr.generic_depths(*X.shape[::-1])).e_s
            _assert_ratio(case, "sklearn weights", float(np.max(np.abs(got["weights"][i] - w_sk)))
                          / (2 * eps * scale / GAMMA), i)
    return refs


def _jorion_s1(engine, batch, N):
    """Jorion's S1 of the same batch where Jorion runs (m > N + 2) and N <= 1536, else None."""
    if batch.rolling_window - 1 <= N + 2 or N > 1536:
        return None
    j = engine.jorion(batch, outputs=("S1",))
    return j["S1"]


# ------------------------------------------------------------------------------------------------- shape sweeps
COLUMNS = [1, 2, 31, 32, 33, 63, 64, 65, 127, 128, 129, 255, 256, 257, 500, 1536, 3072]


@pytest.mark.parametrize("N", COLUMNS)
def test_columns(engine, N):
    """Columns at the 2-column, 64-column (beta_ loop), 32-lane and 8-warp (trace / Frobenius loops) edges, up to
    chol_max_assets(1) = 3072.  m = N + 40 lets Jorion run on the same batch up to N = 1536."""
    n = N + 41 if N <= 1536 else 252
    W = 4 if N < 1024 else 2
    mkt = _market(N, n + W + 2, seed=1000 + N)
    _upload(engine, mkt)
    D = n + W + 2
    batch = _plan(mkt, n, range(D - W, D))
    got, gw = run(f"columns N={N}", engine, batch)
    assert gw["add_blocks"] == 0                      # fewer windows than the block-reuse minimum
    jo = _jorion_s1(engine, batch, N)
    assert (jo is not None) == (N <= 1536)
    windows = range(W) if N < 1024 else (0, W - 1)
    check(f"columns N={N}", engine, mkt, batch, got, windows, jorion=jo)


@pytest.mark.parametrize("K", [2, 3, 15, 16, 17, 31, 33, 251])
def test_rows(engine, K):
    """The row-pair loop with and without its single last row, and warps with no rows (K < 16)."""
    N, W = 40, 4
    n = K + 1
    D = n + W + 2
    mkt = _market(N, D, seed=2000 + K)
    _upload(engine, mkt)
    batch = _plan(mkt, n, range(D - W, D))
    got, _ = run(f"rows K={K}", engine, batch)
    check(f"rows K={K}", engine, mkt, batch, got, range(W), jorion=_jorion_s1(engine, batch, N))


@pytest.mark.parametrize("N,n", [(64, 33), (257, 121)])
def test_more_assets_than_returns(engine, N, n):
    """N >= m: C is singular and only rho > 0 makes the system definite, the regime the estimator exists for."""
    W = 4
    D = n + W + 2
    mkt = _market(N, D, seed=3000 + N)
    _upload(engine, mkt)
    batch = _plan(mkt, n, range(D - W, D))
    got, _ = run(f"N={N} >= m={n - 1}", engine, batch)
    assert np.all(got["scalars"][:, SC["shrinkage"]] > 0)
    check(f"N={N} >= m={n - 1}", engine, mkt, batch, got, range(W), sklearn=True)


# ------------------------------------------------------------------------------------------------- clipping
@pytest.mark.parametrize("N,n,W,step,min_clipped", [(20, 121, 40, 1, 10), (256, 1001, 16, 60, 8)])
def test_clipped_windows(engine, N, n, W, step, min_clipped):
    """i.i.d. equal-volatility returns: many windows clip to s = 1 exactly.  Their weights are finite, status 0 and
    mean / (gamma mu) to the bound; S1 is mu m I.  With the condition estimate on, anorm1 = mu m and rcond = 1 to a
    few ulps, and every other output keeps its bits.  At N = 256 the windows are 60 dates apart with m = 1000: i.i.d.
    windows clip more often the more returns they have."""
    D = n + W * step + 2
    mkt = _market(N, D, seed=4000 + N, iid=True, rf_mode="constant")
    _upload(engine, mkt)
    batch = _plan(mkt, n, [D - 1 - step * k for k in range(W)][::-1])
    case = f"clipped N={N}"
    got, _ = run(case, engine, batch, consecutive=step == 1)
    refs = check(case, engine, mkt, batch, got, range(W), jorion=_jorion_s1(engine, batch, N))
    sure = [i for i, r in refs.items() if r.clipped and float((r.beta - r.delta) / r.delta) > 1e3 * r.e_s]
    assert len(sure) >= min_clipped, len(sure)
    s = got["scalars"][:, SC["shrinkage"]]
    for i in sure:
        assert s[i] == 1.0 and got["status"][i] == 0 and np.all(np.isfinite(got["weights"][i]))
        mean_over_mu = refs[i].t / (LD(refs[i].m) * LD(GAMMA) * refs[i].mu)
        x, eps = refs[i].solution()
        assert lr.ratio(got["weights"][i], mean_over_mu, (eps + 2 * U) * float(np.max(np.abs(mean_over_mu)))) < 1
    engine.set_condition_estimate(True)
    try:
        engine.solve_work()
        cg = engine.shrinkage(batch, outputs=OUTS)
        assert engine.solve_work() == {"factored": W, "chained": 0}
    finally:
        engine.set_condition_estimate(False)
    for k in OUTS:
        if k == "scalars":
            assert np.array_equal(cg[k][:, :SC["anorm1"]], got[k][:, :SC["anorm1"]])
        else:
            assert np.array_equal(cg[k], got[k]), k
    m = np.float64(n - 1)
    for i in sure:
        assert cg["scalars"][i, SC["anorm1"]] == np.float64(got["scalars"][i, SC["mu"]]) * m
        assert abs(cg["scalars"][i, SC["rcond"]] - 1.0) <= 8 * np.spacing(1.0), cg["scalars"][i, SC["rcond"]]


@pytest.mark.parametrize("log2_gap,seed", [(20, 5020), (40, 5042)])
def test_near_clipped_windows(engine, log2_gap, seed):
    """s = 1 - 2^-k from a common factor mixed into i.i.d. returns, its scale found by bisection on the reference.
    The weights stay within a bound that rests on ds |C|, not on the relative error of 1 - s."""
    N, n = 20, 121
    D = n + 3
    K = n - 1
    rng = np.random.default_rng(seed)
    mkt = _market(N, D, seed=seed, rf_mode="constant")
    R = lr.iid_returns(D, N, rng)
    f = rng.standard_normal(K) * 0.01
    rows = gr.daily_return_rows(D - 1, n)

    def window_X(c):
        Rc = R.copy()
        Rc[rows] = lr.mixed_returns(R[rows], f, c)
        P = 100.0 * np.exp(np.cumsum(Rc, axis=0))
        return np.log(P[rows] / P[rows - 1]), Rc

    def s_of(c):
        X, _ = window_X(c)
        Xc = X - X.mean(axis=0)
        return lr.LWRef(X, Xc.T @ Xc).s

    assert s_of(0.0) == 1                                  # this seed's window clips without the factor
    target = 1.0 - 2.0 ** -log2_gap
    lo, hi = 0.0, 1.0
    for _ in range(200):
        mid = 0.5 * (lo + hi)
        if mid in (lo, hi):
            break
        lo, hi = (mid, hi) if s_of(mid) >= target else (lo, mid)
    _set_log_returns(mkt, window_X(0.5 * (lo + hi))[1])
    _upload(engine, mkt)
    batch = _plan(mkt, n, [D - 1])
    case = f"near-clipped 1-2^-{log2_gap}"
    got, _ = run(case, engine, batch)
    refs = check(case, engine, mkt, batch, got, [0], jorion=_jorion_s1(engine, batch, N))
    gap = float(1 - refs[0].s)
    assert abs(np.log2(gap) + log2_gap) < 0.5, gap


def test_one_asset(engine):
    """N = 1: sklearn's shrinkage is 0 whatever delta rounds to; the weight is t / (gamma C)."""
    n, W = 60, 64
    D = n + W + 2
    mkt = _market(1, D, seed=6001)
    _upload(engine, mkt)
    batch = _plan(mkt, n, range(D - W, D))
    got, _ = run("one asset", engine, batch, consecutive=True)
    assert np.all(got["scalars"][:, SC["shrinkage"]] == 0.0)
    assert not got["status"].any() and np.all(np.isfinite(got["weights"]))
    check("one asset", engine, mkt, batch, got, range(W))


# ------------------------------------------------------------------------------------------------- routes
def test_weekly_windows(engine):
    """Weekly windows read the resampled rows and their extra_row (the trade date's partial week)."""
    from incorporating_different_sources_b200.windows import plan_weekly_windows
    N, n, W = 24, 60, 12
    D = 7 * n + 40
    mkt = _market(N, D, seed=7001)
    _upload(engine, mkt)
    spec = _spec(N, n, freq="weekly")
    d_idx = [D - 1 - 3 * k for k in range(W)][::-1]
    rows, batch = plan_weekly_windows(spec, mkt.dates, d_idx, mkt.dates, mkt.rf, None, need_hf=False)
    assert np.any(batch.extra_row >= 0)
    engine.set_resampled(rows)
    got, _ = run("weekly", engine, batch)
    a_max = (1.0 + float(mkt.rf.max())) ** (7.0 / 365.0) - 1.0

    def weekly_rows(i):
        # the oracle's rows: the same correctly rounded price ratios, a = (1 + rf)^(gbar/365) - 1 to a few ulp of 1
        _, _, X = bo.daily_statistics(spec, mkt, d_idx[i], np.arange(N))
        a = np.full(X.shape[0], a_max)
        return X, a, 4 * U * (np.abs(X) + 2.0 * a_max + 1.0)
    check("weekly", engine, mkt, batch, got, range(W), rows=weekly_rows)


def test_chunked_batch(engine):
    """A workspace limit of two windows: at least three chunks, windows with different span_days and risk-free rates,
    bit for bit the one-chunk result and within the bound (a wrong window offset of a chunk shows in both)."""
    N, n, W = 33, 62, 9
    D = n + 60
    mkt = _market(N, D, seed=8001)
    _upload(engine, mkt)
    d_idx = [D - 1 - 6 * k - (k % 3) for k in range(W)][::-1]
    batch = _plan(mkt, n, d_idx)
    assert len(set(batch.span_days.tolist())) >= 2
    engine.set_stage_timing(True)
    try:
        engine.stage_times()
        one, _ = run("chunked: one chunk", engine, batch)
        g1 = engine.stage_times()["gram"]["launches"]
        ld, ldS = -(-N // 16) * 16, -(-N // 32) * 32
        per_window = 8 * ((ldS + 8) * ldS + 9 * ld + 16) + 16
        engine.set_workspace_limit(2 * per_window + 64)
        chunked, _ = run("chunked", engine, batch)
        g3 = engine.stage_times()["gram"]["launches"]
    finally:
        engine.set_stage_timing(False)
        engine.set_workspace_limit(24 << 30)
    assert g1 >= 1 and g3 >= 3 * g1, (g1, g3)
    for k in OUTS:
        assert np.array_equal(one[k], chunked[k]), k
    check("chunked", engine, mkt, batch, chunked, range(W))


@pytest.mark.parametrize("reuse", [True, False])
def test_gram_routes(engine, reuse):
    """40 consecutive windows of 251 returns: block Gram tiles reused (reuse minimum 32) or every window from
    scratch; both within the bound, the planner never chains, and two identical calls give the same bits."""
    N, n, W = 64, 252, 40
    D = n + W + 2
    mkt = _market(N, D, seed=9001)
    _upload(engine, mkt)
    batch = _plan(mkt, n, range(D - W, D))
    case = f"gram {'block reuse' if reuse else 'from scratch'}"
    engine.set_reuse_min_windows(32 if reuse else NO_REUSE)
    try:
        got, gw = run(case, engine, batch, consecutive=True)
        again = engine.shrinkage(batch, outputs=OUTS)
        jo = _jorion_s1(engine, batch, N)
    finally:
        engine.set_reuse_min_windows(32)
    assert (gw["add_blocks"] > 0) == reuse, gw
    for k in OUTS:
        assert np.array_equal(got[k], again[k]), k
    check(case, engine, mkt, batch, got, range(W), jorion=jo)


# ------------------------------------------------------------------------------------------------- facade, backtest
def _clipping_market(N, D, seed):
    from incorporating_different_sources_b200.synthetic import generate_market
    mkt = generate_market(N, D, seed=seed, bars_per_day=2, rf_mode="constant")
    _set_log_returns(mkt, lr.iid_returns(D, N, np.random.default_rng(seed)))
    return mkt


def _sk_shrinkage_window(spec, mkt, d, cols):
    from sklearn.covariance import ledoit_wolf
    return bo.shrinkage_window(spec, mkt, d, cols, cov_fn=ledoit_wolf)


def test_facade_on_clipped_window():
    """calculate_shrinkage_portfolio on a window whose intensity clips: clean_weights of sklearn's weights."""
    from incorporating_different_sources_b200 import portfolio_calculations as pc
    N, n = 20, 121
    mkt = _clipping_market(N, n + 40, seed=10002)
    spec = _spec(N, n)
    cols = np.arange(N)
    d = next(d for d in range(n, n + 40) if _sk_shrinkage_window(spec, mkt, d, cols)["shrinkage"] == 1.0)
    md = mkt.market_data()
    ts = pd.Timestamp(mkt.dates[d])
    w = pc.calculate_shrinkage_portfolio(spec, ts, md["stock_prices_df"].loc[:ts], md["risk_free_rate_df"])
    ref = _sk_shrinkage_window(spec, mkt, d, cols)["weights"]
    order = [mkt.tickers[c] for c in cols]
    got = w.loc[order, "Weight"].to_numpy()
    assert np.all(np.isfinite(got))
    assert np.array_equal(got, bo.clean_weights(ref))


def test_backtest_on_clipping_market(engine, monkeypatch):
    """A short daily shrinkage backtest on an i.i.d. market where windows clip: the loop receives finite weights
    equal to the oracle's clean weights, and the returns are finite."""
    from incorporating_different_sources_b200.backtest import backtest_portfolio
    from tests import _loop_ref as lpr
    N, n = 20, 121
    mkt = _clipping_market(N, n + 40, seed=10002)
    md = mkt.market_data()
    spec = _spec(N, n)
    start, end = mkt.dates[n + 5], mkt.dates[n + 30]
    seen = {}
    real = engine.backtest_loop

    def spy(reb_rows, weights, *args, **kw):
        seen.update(reb=np.array(reb_rows), W=np.array(weights))
        return real(reb_rows, weights, *args, **kw)

    monkeypatch.setattr(engine, "backtest_loop", spy)
    res = backtest_portfolio(spec, pd.Timestamp(start), pd.Timestamp(end), md, engine=engine)
    orc = lpr.oracle_inputs(spec, mkt, md, start, end)
    clipped = sum(_sk_shrinkage_window(spec, mkt, int(r), np.arange(N))["shrinkage"] == 1.0 for r in orc.reb_row)
    assert clipped >= 3, clipped
    assert np.array_equal(seen["reb"], orc.reb_row)
    assert np.all(np.isfinite(seen["W"]))
    assert np.max(np.abs(seen["W"] - orc.W)) <= 1e-12
    assert np.all(np.isfinite(res["portfolio_simple_returns_series"].to_numpy()))
