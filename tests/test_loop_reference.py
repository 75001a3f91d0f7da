"""The loop-body restatement (tests/_loop_ref.py) on the CPU: pinned on the reference's own backtests
(tests/golden/bt_*.npz), accurate against exact rational arithmetic, its bound honoured by float64 in any summation
order, and far exceeded by each seeded fault on the cases tests/test_gpu_loop.py runs on the kernel."""
import glob
import json
import os
from fractions import Fraction

import numpy as np
import pytest

from incorporating_different_sources_b200.synthetic import generate_market
from tests import _loop_ref as lr
from tests.golden.make_backtest_golden import apply_damage
from tests.test_gpu_backtest import _close

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
NAMES = sorted(os.path.basename(p)[:-4] for p in glob.glob(os.path.join(GOLD, "bt_*.npz")))
REPORT = {}                 # line -> text, printed at the end of the module


@pytest.fixture(scope="module", autouse=True)
def report(request):
    lr.require_extended_precision()
    yield
    capman = request.config.pluginmanager.getplugin("capturemanager")
    with capman.global_and_fixture_disabled():
        print("\nloop-body restatement:")
        for k in sorted(REPORT):
            print(f"  {k:44s} {REPORT[k]}")


def golden_inputs(name):
    z = np.load(os.path.join(GOLD, name + ".npz"))
    meta = json.loads(str(z["meta"]))
    mkt = generate_market(**meta["market"])
    md = apply_damage(mkt.market_data(), meta.get("damage"))
    if meta.get("damage"):
        mkt.prices = md["stock_prices_df"].to_numpy(dtype=np.float64).copy()      # the oracle reads the same prices
    return lr.oracle_inputs(meta["spec"], mkt, md, meta["start"], meta["end"]), z


@pytest.mark.parametrize("name", NAMES)
def test_restatement_reproduces_reference_backtest(name):
    inp, z = golden_inputs(name)
    ref = lr.restate(inp)
    r, t, m = (np.asarray(x, dtype=np.float64) for x in (ref.returns, ref.turnover, ref.metrics))
    _close(r, z["returns"])
    _close(t, z["turnover"])
    _close(m, z["metrics"])
    # the largest |difference| as a share of _close's tolerance (1e-9 max|b| + 1e-13)
    share = max(float(np.nanmax(np.abs(a - z[k])) / (1e-9 * np.nanmax(np.abs(z[k])) + 1e-13))
                for a, k in ((r, "returns"), (t, "turnover"), (m, "metrics")) if len(a))
    REPORT[f"golden {name}"] = (f"reproduced: {len(r)} returns, {len(t)} turnovers, {m.shape[0]} x 5 metrics, "
                                f"max |diff| = {share:.1e} x tolerance")


def _frac(x):
    return Fraction(*np.longdouble(x).as_integer_ratio())


def test_longdouble_reference_against_exact_fractions():
    """~20 days of drift in three segments and a tail, a universe that changes at every rebalance, sum w != 1, a price
    hole in a held column: the longdouble evaluation is within 2**-11 of the bound of the exact one."""
    inp = lr.case(6, 30, [2, 9, 10, 21], 27, seed=11, bps=1000.0, holes=[(3, 4, 1)])
    assert any(abs(inp.W[s].sum() - 1) > 0.1 for s in range(inp.R))
    assert np.isnan(inp.prices).any()
    ref = lr.restate(inp)
    ex = lr.restate(inp, lr.FRACTION)
    worst = 0.0
    for got, exact, bnd in ((ref.returns, ex.returns, ref.b_returns), (ref.turnover, ex.turnover, ref.b_turnover),
                            (ref.metrics[:, 2:].ravel(), ex.metrics[:, 2:].ravel(), ref.b_metrics[:, 2:].ravel())):
        for g, e, b in zip(got, exact, bnd):
            if isinstance(e, float) and np.isnan(e):
                assert np.isnan(float(g))
                continue
            worst = max(worst, float(abs(_frac(g) - e)) / b)
    assert np.array_equal(ref.metrics[:, :2].astype(float), ex.metrics[:, :2].astype(float), equal_nan=True)
    REPORT["exact check longdouble |E| / bound"] = f"{worst:.2e}"
    assert worst < 2.0 ** -11


@pytest.fixture(scope="module")
def wide():
    """N = 2048 with a 250-day segment, a mask that changes at each rebalance and a 9-day tail."""
    inp = lr.case(2048, 262, [1, 251, 252], 261, seed=21, scale=1.0, bps=15.0)
    return inp, lr.restate(inp)


@pytest.mark.parametrize("order", ["kernel", "forward", "reverse", "random"])
def test_float64_honours_bound_in_any_summation_order(wide, order):
    inp, ref = wide
    f = lr.restate(inp, lr._F64(order, seed=5))
    r = lr.ratios((f.returns, f.turnover, f.metrics), ref)
    REPORT[f"float64 {order} order, N = 2048"] = " ".join(f"{k}={v:.2g}" for k, v in r.items())
    assert max(r.values()) < 1.0, r


# faults and the case of tests/test_gpu_loop.py that shows each (the same builders, the same seeds)
FAULT_CASES = {
    "drift_from_rebalance_day": "weekly",
    "held_is_new_member": "changing",
    "no_rf_leg": "weekly",
    "rf_365": "weekly",
    "no_rf_turnover": "changing",
    "cost_day_after": "monthly",
    "nan_weight_counts": "holes",
    "capsum_all_columns": "changing",
    "max_warp0_only": "n257",
}


def fault_case(name):
    if name == "holes":
        return lr.hole_case()
    if name == "changing":
        return lr.width_case(500)
    if name == "n257":
        return lr.width_case(257)
    return lr.SEGMENT_CASES[name]()


@pytest.mark.parametrize("fault", lr.FAULTS)
def test_bound_catches_seeded_fault(fault):
    inp = fault_case(FAULT_CASES[fault])
    ref = lr.restate(inp)
    bad = lr.restate(inp, fault=fault)
    r = lr.ratios((bad.returns, bad.turnover, bad.metrics), ref)
    worst = max(r.values())
    REPORT[f"fault {fault}"] = f"{worst:.3g} x bound ({FAULT_CASES[fault]} case, {max(r, key=r.get)})"
    assert worst >= 100.0, r
