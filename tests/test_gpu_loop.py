"""The backtest loop body (loop_kernels.cu through BayesEngine.backtest_loop) on its own, every output held to the
a-priori bound of tests/_loop_ref.py (max_long / max_short bit for bit): widths at the kernel's lane, warp and
register-slot edges up to the 2,048-asset limit, every segment shape, changing and one-stock universes, price holes in
held columns, poisoned columns the loop must never read, every input / output route, and the loop level of
``backtest_portfolio`` at ~700 tickers against the oracle.

NaN weights of members at a rebalance date are not tested: they only arise from a failed solve, and
``backtest_portfolio`` raises on the window's status before the loop runs."""
import numpy as np
import pandas as pd
import pytest

from tests import _loop_ref as lr
from tests.test_gpu_backtest import _close

pytestmark = pytest.mark.gpu
WORST = {}                  # case -> output -> worst |E| / bound (printed at the end of the module)


@pytest.fixture(scope="module")
def engine(request):
    from incorporating_different_sources_b200.engine import BayesEngine
    lr.require_extended_precision()
    eng = BayesEngine(0)
    yield eng
    eng.close()
    if WORST:
        with request.config.pluginmanager.getplugin("capturemanager").global_and_fixture_disabled():
            print("\nworst |E| / bound per case:")
            for name, d in WORST.items():
                print(f"  {name:30s} " + " ".join(f"{k}={v:.3g}" for k, v in d.items()))


def run(eng, inp: lr.LoopInputs, weights=None, **kw):
    eng.upload_market(inp.prices, inp.rf_row, caps=inp.caps)
    return eng.backtest_loop(inp.reb_row, inp.W if weights is None else weights, distance_scale=inp.scale,
                             turnover_cost_bps=inp.bps, member=inp.member, last_row=inp.last_row, **kw)


def check(name, inp, got, ref=None):
    ref = lr.restate(inp) if ref is None else ref
    r = lr.ratios(got, ref)
    WORST[name] = r
    assert max(r.values()) < 1.0, f"{name}: {r}"


def same_bits(a, b):
    a, b = (np.ascontiguousarray(x, dtype=np.float64) for x in (a, b))
    return a.shape == b.shape and np.array_equal(a.view(np.int64), b.view(np.int64))


@pytest.mark.parametrize("N", lr.WIDTHS)
def test_widths(engine, N):
    inp = lr.width_case(N)
    check(f"N={N}", inp, run(engine, inp))


def test_2049_assets_refused(engine):
    """The kernel holds 8 assets per thread in registers: one more than 8 x 256 is refused on the host, as invalid input
    (ValueError, the engine's mapping of BP_ERR_INVALID), before anything is launched."""
    inp = lr.case(2049, 12, [2, 5], 9, seed=7)
    engine.upload_market(inp.prices, inp.rf_row, caps=inp.caps)
    n = engine.launch_count
    with pytest.raises(ValueError, match="at most 2048 assets"):
        engine.backtest_loop(inp.reb_row, inp.W, 1.0, 15.0, member=inp.member, last_row=inp.last_row)
    assert engine.launch_count == n


@pytest.mark.parametrize("name", list(lr.SEGMENT_CASES))
def test_segments_and_universes(engine, name):
    inp = lr.SEGMENT_CASES[name]()
    check(name, inp, run(engine, inp))


def test_price_holes_in_held_columns(engine):
    """A halt on the day after a rebalance, a two-day halt and a mid-segment delisting: the column's weight turns NaN
    for the rest of the segment, drops out of every sum and counts 0 in the turnover.  The same case treated as if the
    weight kept counting misses the bound by far (tests/test_loop_reference.py), so the NaN path is what is checked."""
    inp = lr.hole_case()
    check("price_holes", inp, run(engine, inp))


@pytest.mark.parametrize("name", ["N=500", "N=2048", "price_holes"])
def test_non_member_columns_are_never_read(engine, name):
    inp = lr.hole_case() if name == "price_holes" else lr.width_case(int(name[2:]))
    clean = run(engine, inp)
    bad = lr.poisoned(inp)
    assert np.isnan(bad.prices).any() and np.isinf(bad.prices).any() and np.isnan(bad.W).any()
    dirty = run(engine, bad)
    for a, b in zip(clean, dirty):
        assert same_bits(a, b)


def test_routes_give_the_same_bits(engine):
    import torch
    inp = lr.width_case(1793)
    base = run(engine, inp)
    check("routes N=1793", inp, base)
    again = engine.backtest_loop(inp.reb_row, inp.W, inp.scale, inp.bps, member=inp.member, last_row=inp.last_row)
    on_dev = engine.backtest_loop(inp.reb_row, torch.tensor(inp.W, device="cuda"), inp.scale, inp.bps,
                                  member=inp.member, last_row=inp.last_row)
    dev_out = engine.backtest_loop(inp.reb_row, inp.W, inp.scale, inp.bps, member=inp.member, last_row=inp.last_row,
                                   device_out=True)
    dev_out = [t.cpu().numpy() for t in dev_out]
    # the same columns selected from a pool that holds them shuffled among others
    rng = np.random.default_rng(3)
    extra = 211
    perm = rng.permutation(inp.N + extra)
    D = inp.prices.shape[0]
    pool_p = rng.uniform(1.0, 2.0, (D, inp.N + extra))
    pool_c = rng.uniform(1.0, 2.0, (D, inp.N + extra))
    pool_p[:, perm[:inp.N]] = inp.prices
    pool_c[:, perm[:inp.N]] = inp.caps
    engine.upload_pool(pool_p, inp.rf_row, caps=pool_c)
    try:
        engine.select_market(perm[:inp.N], 0, D, 0, 0)
        pooled = engine.backtest_loop(inp.reb_row, inp.W, inp.scale, inp.bps, member=inp.member, last_row=inp.last_row)
    finally:
        engine.upload_pool(None, None)
    for other in (again, on_dev, dev_out, pooled):
        for a, b in zip(base, other):
            assert same_bits(a, b)


# ------------------------------------------------------------------------------------------------- loop level
@pytest.fixture(scope="module")
def wide_market():
    """~700 tickers, 480 days: one late listing (NaN prices until row 445) and one mid-month delisting (NaN prices from
    row 457 on) of the stock with the largest caps, which every top-300..500 universe holds."""
    from incorporating_different_sources_b200.synthetic import generate_market
    mkt = generate_market(700, 480, seed=4242)
    order = np.argsort(-mkt.caps[440])
    late, gone = int(order[1]), int(order[0])
    mkt.prices[:445, late] = np.nan
    mkt.prices[457:, gone] = np.nan
    return mkt, mkt.market_data(), gone


SPECS = {
    "jeffreys_monthly": dict(weighting_strategy="jeffreys", size=300, risk_aversion=1000, turnover_cost=15,
                             rebalancing_frequency="monthly", rolling_window=400, rolling_window_frequency="daily",
                             mcm_scaling=None, display_name="Jeffreys"),
    "conjugate_weekly": dict(weighting_strategy="conjugate_hf_vix_vw", size=400, risk_aversion=500, turnover_cost=15,
                             rebalancing_frequency="weekly", rolling_window=420, rolling_window_frequency="daily",
                             mcm_scaling=1, display_name="Conjugate HF-VIX VW"),
    "vw_daily": dict(weighting_strategy="vw", size=500, risk_aversion=None, turnover_cost=15,
                     rebalancing_frequency="daily", rolling_window=20, rolling_window_frequency="daily",
                     mcm_scaling=None, display_name="VW"),
}


@pytest.mark.parametrize("name", list(SPECS))
def test_loop_level_at_scale(engine, wide_market, monkeypatch, name):
    from incorporating_different_sources_b200.backtest import backtest_portfolio
    mkt, md, gone = wide_market
    spec = SPECS[name]
    start, end = mkt.dates[430], mkt.dates[479]
    seen = {}
    real = engine.backtest_loop

    def spy(reb_rows, weights, distance_scale, turnover_cost_bps, member=None, last_row=None, device_out=False):
        seen.update(reb=np.array(reb_rows), W=np.array(weights), scale=distance_scale, bps=turnover_cost_bps,
                    member=np.array(member), last_row=last_row)
        return real(reb_rows, weights, distance_scale, turnover_cost_bps, member=member, last_row=last_row,
                    device_out=device_out)

    monkeypatch.setattr(engine, "backtest_loop", spy)
    res = backtest_portfolio(spec, pd.Timestamp(start), pd.Timestamp(end), md, engine=engine)
    got = (res["portfolio_simple_returns_series"].to_numpy(), res["portfolio_turnover_series"].to_numpy(),
           res["portfolio_weights_metrics_df"].to_numpy())
    orc = lr.oracle_inputs(spec, mkt, md, start, end)
    assert np.array_equal(seen["reb"], orc.reb_row) and seen["last_row"] == orc.last_row
    assert np.array_equal(seen["member"], orc.member)
    assert orc.member[:, gone].any() and not orc.member[-1, gone]          # held, then delisted
    held_w = np.abs(orc.W).max(axis=1, keepdims=True)
    assert np.all(np.abs(seen["W"] - orc.W) <= 1e-9 * held_w)
    assert seen["scale"] == orc.scale and seen["bps"] == orc.bps
    rec = lr.LoopInputs(orc.prices, orc.caps, orc.rf_row, seen["reb"], seen["W"], seen["member"], seen["last_row"],
                        float(seen["scale"]), float(seen["bps"]))
    check(f"loop level {name}", rec, got)
    ref = lr.restate(orc)
    for a, b in zip(got, (ref.returns, ref.turnover, ref.metrics)):
        _close(a, np.asarray(b, dtype=np.float64))
