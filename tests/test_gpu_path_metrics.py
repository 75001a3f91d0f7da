"""path_metrics_kernel on its own (bp_path_metrics through evaluation.path_metrics), every statistic of every series
held to the a-priori bound of the longdouble reference (tests/_eval_ref.py): lengths at the edges of the chunked scan
(T = 2 .. 100,003, a multiple of 256, one above, a last thread holding one return), ensembles of 1 to 3,000 series,
drawdowns placed against the chunk boundaries, -100 % days and adjusted insolvencies, empty conditional selections,
ill-conditioned moments, constant series, and years from 2/365 to 40.  Best and Worst Day, and a zero drawdown, must
match bit for bit; NaN and +-inf must sit where the reference has them."""
import numpy as np
import pytest

from incorporating_different_sources_b200 import evaluation as ev
from tests import _eval_ref as er

pytestmark = pytest.mark.gpu

WORST = {}                 # statistic -> (worst |E| / bound, case)


@pytest.fixture(scope="module", autouse=True)
def report(request):
    er.require_extended_precision()
    yield
    if WORST:
        capman = request.config.pluginmanager.getplugin("capturemanager")
        with capman.global_and_fixture_disabled():
            print("\nworst |E| / bound per statistic:")
            for name in er.NAMES:
                if name in WORST:
                    print(f"  {name:18s} {WORST[name][0]:.3g}  ({WORST[name][1]})")


def _check(name, r, x, years):
    """Run one call and hold every series to its bound; returns the kernel's [P][16] output."""
    got = ev.path_metrics(r, x, years)
    assert got.shape == (len(r), 16)
    for p in range(len(r)):
        ref = er.restate(r[p], x[p], years)
        rat = er.ratios(got[p], ref)
        for k, v in enumerate(rat):
            if np.isfinite(v) and v > WORST.get(er.NAMES[k], (-1.0,))[0]:
                WORST[er.NAMES[k]] = (float(v), name)
        bad = {er.NAMES[k]: (got[p, k], float(ref.values[k]), ref.bound[k]) for k in np.nonzero(~(rat < 1.0))[0]}
        assert not bad, f"{name}, series {p} of {len(r)}: (kernel, reference, bound) {bad}"
    return got


def _run(name):
    with np.errstate(all="ignore"):
        calls = er.CASES[name]()
    return [(r, x, years, _check(name, r, x, years)) for r, x, years in calls]


@pytest.mark.parametrize("name", [n for n in er.CASES if n.startswith(("length_", "ensemble_", "dd_across", "dd_inside",
                                                                       "moments_", "years"))])
def test_statistics_within_bound(name):
    _run(name)


@pytest.mark.parametrize("T", [257, 512, 4149])
def test_drawdown_shapes(T):
    """Peak at index 0 / trough at T - 1, a curve declining from the first day (its peak is W_0, not 1), a global peak
    and a trough in the last return, and a curve that never falls (Max. DD exactly 0)."""
    (r, x, _, got), = _run(f"dd_shapes_{T}")
    dd = got[:, er.K["Max. DD"]]
    assert dd[4] == 0.0 and np.isinf(got[4, er.K["Calmar"]])
    w = np.cumprod(1.0 + r[1])
    assert abs(dd[1] - (w[-1] / w[0] - 1.0)) < 1e-9 < abs(dd[1] - (w[-1] - 1.0))


@pytest.mark.parametrize("T", [257, 4149])
def test_wipe_out(T):
    """A -100 % day: total, CAGR and drawdown exactly -1, Calmar -1; the empty chunks after it (0 * -inf = NaN in the
    combine) leak nothing."""
    (r, x, _, got), = _run(f"wipe_out_{T}")
    for p in (0, 1):
        assert got[p, er.K["Cum. Return"]] == -1.0 and got[p, er.K["CAGR"]] == -1.0
        assert got[p, er.K["Max. DD"]] == -1.0 and got[p, er.K["Calmar"]] == -1.0
        assert np.all(np.isfinite(got[p]))


@pytest.mark.parametrize("T", [257, 4149])
def test_adjusted_insolvency(T):
    """After adjust_returns the wealth changes sign once and stays constant: negative in the first series (base < 0
    turns an empty chunk's -inf into +inf in the combine), tiny and positive in the second."""
    (r, x, _, got), = _run(f"insolvent_{T}")
    w = np.cumprod(1.0 + r, axis=1)[:, -1]
    assert w[0] < 0 < w[1] < 1e-3
    assert got[0, er.K["Cum. Return"]] < -1.0 and got[0, er.K["Max. DD"]] < -1.0
    assert np.all(np.isfinite(got[:, :er.K["Calmar"] + 1]))


@pytest.mark.parametrize("T", [40, 513, 4149])
def test_conditional_statistics(T):
    """No losing day (Avg. Loss NaN, Max. DD 0), no winning day (Avg. Win NaN), all zeros (NaN averages, Sharpe,
    Sortino, skew, kurtosis; zero volatility), zeros mixed in (Avg. Return skips them), no negative excess
    (Sortino +inf)."""
    (r, x, _, got), = _run(f"conditional_{T}")
    K = er.K
    assert np.isnan(got[0, K["Avg. Loss"]]) and got[0, K["Max. DD"]] == 0.0
    assert np.isnan(got[1, K["Avg. Win"]])
    assert all(np.isnan(got[2, K[k]]) for k in ("Avg. Loss", "Avg. Return", "Avg. Win", "Sharpe", "Sortino", "skew",
                                                "kurtosis", "sharpe_per_period", "Calmar"))
    assert got[2, K["Ann. Vol."]] == 0.0 and got[2, K["Cum. Return"]] == 0.0 and got[2, K["Max. DD"]] == 0.0
    nz = r[3][r[3] != 0]
    assert abs(got[3, K["Avg. Return"]] - nz.mean()) < 1e-12 * np.abs(nz).mean()
    assert got[4, K["Sortino"]] == np.inf


@pytest.mark.parametrize("T,v", er.CONSTANTS, ids=[f"{T}x{v:.3g}" for T, v in er.CONSTANTS])
def test_constant_excess_series(T, v):
    """Constant excess returns: skewness and kurtosis are NaN (the exact m2 is 0) whether or not the kernel's block-sum
    mean is exact; Sharpe is +-inf, or a finite value of the same sign at least as large as the mean error allows."""
    (r, x, _, got), = _run(f"constant_{T}_{v:.3g}")
    assert np.isnan(got[0, er.K["skew"]]) and np.isnan(got[0, er.K["kurtosis"]])
    assert np.sign(got[0, er.K["Sharpe"]]) == np.sign(v)
