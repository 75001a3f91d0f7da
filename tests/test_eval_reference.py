"""The path-metrics restatement (tests/_eval_ref.py) on the CPU: pinned on oracle/eval_oracle.path_row, accurate
against exact rational arithmetic, its bound honoured by a float64 emulation of the kernel in its own order and in
others, and far exceeded (or an exact output broken) by each seeded fault on the cases tests/test_gpu_path_metrics.py
runs on the kernel."""
import warnings
from fractions import Fraction

import numpy as np
import pandas as pd
import pytest

from incorporating_different_sources_b200 import evaluation as ev
from oracle import eval_oracle as eo
from tests import _eval_ref as er

REPORT = {}                 # line -> text, printed at the end of the module


@pytest.fixture(scope="module", autouse=True)
def report(request):
    er.require_extended_precision()
    yield
    capman = request.config.pluginmanager.getplugin("capturemanager")
    with capman.global_and_fixture_disabled():
        print("\npath-metrics restatement:")
        for k in sorted(REPORT):
            print(f"  {k:44s} {REPORT[k]}")


def _calls(name):
    with np.errstate(all="ignore"):
        return er.CASES[name]()


def test_names_follow_the_metric_rows():
    assert list(er.NAMES) == ev.METRIC_ROWS


@pytest.mark.parametrize("P,T", [(8, 4149), (6, 257), (4, 2), (4, 513)])
def test_reference_matches_oracle(P, T):
    """The oracle (NumPy / scipy in float64) is one more summation order: on well-conditioned series it sits within the
    bound of the longdouble reference, and skewness / kurtosis / NaNs agree."""
    r, x = er.series(P, T, 77 + T)
    r[1, ::9] = 0.0
    idx = pd.bdate_range("2007-01-03", periods=T)
    years = (idx[-1] - idx[0]).days / 365
    worst = 0.0
    for p in range(P):
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            row = eo.path_row(r[p], x[p], idx)
        rat = er.ratios(row, er.restate(r[p], x[p], years))
        worst = max(worst, float(rat.max()))
        assert rat.max() < 1.0, (p, {er.NAMES[k]: rat[k] for k in np.nonzero(rat >= 1)[0]})
    REPORT[f"oracle vs reference, T = {T}"] = f"worst |E| / bound {worst:.2g}"


@pytest.mark.parametrize("name", ["length_2", "dd_shapes_exact", "wipe_out_exact", "insolvent_exact", "conditional_40",
                                  "moments_exact", "constant_exact"])
def test_longdouble_reference_against_exact_arithmetic(name):
    """At small T, Fractions with sqrt / pow from mpmath at 256 bits: the longdouble values are within 2**-10 of their
    bound of the exact ones, and NaN, +-inf and the exact outputs agree."""
    calls = {
        "dd_shapes_exact": lambda: er.dd_shapes(40)(),
        "wipe_out_exact": lambda: er.wipe_out(33)(),
        "insolvent_exact": lambda: er.insolvent(30, 20)(),
        "moments_exact": lambda: er.moments(41)(),
        "constant_exact": lambda: er.constant_case(37, 0.1)(),
    }.get(name, lambda: _calls(name))()
    worst = 0.0
    for r, x, years in calls:
        for p in range(len(r)):
            ref = er.restate(r[p], x[p], years)
            ex = er.restate(r[p], x[p], years, er.EXACT)
            for k in range(16):
                v, e, b = ref.values[k], ex.values[k], ref.bound[k]
                fe = float(e)
                if np.isnan(fe) or np.isinf(fe) or b == 0:
                    assert float(v) == fe or (np.isnan(float(v)) and np.isnan(fe)), (p, er.NAMES[k], v, e)
                elif np.isfinite(b):
                    err = abs(Fraction(*np.longdouble(v).as_integer_ratio()) - e)
                    worst = max(worst, float(err) / b)
    REPORT[f"exact check {name}"] = f"longdouble |E| / bound {worst:.2e}"
    assert worst < 2.0 ** -10


@pytest.mark.parametrize("order", ["kernel", "forward", "random"])
@pytest.mark.parametrize("name", ["length_2", "length_257", "length_4149", "length_65537", "dd_across_chunks_513",
                                  "dd_inside_chunk_4149", "dd_shapes_257", "wipe_out_257", "insolvent_257",
                                  "conditional_513", "moments_4149", "constant_4149_0.1", "constant_601_0.0003",
                                  "years"])
def test_float64_honours_bound_in_any_order(name, order):
    worst = np.zeros(16)
    for r, x, years in _calls(name):
        for p in range(len(r)):
            ref = er.restate(r[p], x[p], years)
            rat = er.ratios(er.kernel_f64(r[p], x[p], years, order=order, seed=p), ref)
            worst = np.maximum(worst, rat)
            assert rat.max() < 1.0, (p, {er.NAMES[k]: rat[k] for k in np.nonzero(rat >= 1)[0]})
    REPORT[f"float64 {order:7s} {name}"] = f"worst {worst.max():.2g} ({er.NAMES[int(worst.argmax())]})"


@pytest.mark.parametrize("T,v", [(4149, 0.1), (257, 3e-4), (601, 3e-4)])
def test_kernel_mean_of_a_constant_is_off_and_the_old_rule_gives_a_skew(T, v):
    """The kernel's block-sum mean of these constants is 1 to 3 ulp off, so x2 / n = delta^2 > 0: without the flat rule
    on the corrected m2 the kernel reports skew = +-1 and kurtosis = 1; with it, NaN."""
    x = np.full(T, v)
    r = np.zeros(T)
    mean = er.kernel_sum(x) / T
    assert mean != v
    old = er.kernel_f64(r, x, 1.0, fault="no_flat_rule")
    assert abs(old[er.K["skew"]]) == 1.0 and old[er.K["kurtosis"]] == 1.0
    new = er.kernel_f64(r, x, 1.0)
    assert np.isnan(new[er.K["skew"]]) and np.isnan(new[er.K["kurtosis"]])


def test_flat_rule_claims_nothing_near_the_threshold():
    """Between 10**-3 and 10**3 times scipy's threshold the two summation orders may disagree: no claim; below it NaN,
    above it a bounded value."""
    rng = np.random.default_rng(3)
    T = 600
    ulp = np.spacing(0.1)
    one_ulp = np.full(T, 0.1)
    one_ulp[rng.integers(T)] += ulp
    series = {"nan": one_ulp,                                                   # m2 ~ ulp^2 / T
              "free": 0.1 + ulp * rng.integers(-2, 3, T),                       # m2 ~ 2 ulp^2
              "bounded": 0.1 + 1e-13 * rng.standard_normal(T)}
    thr = (er.EPS * 0.1) ** 2
    seen = set()
    for kind, x in series.items():
        m2 = float(np.var(x.astype(np.longdouble)))
        assert kind == ("nan" if m2 <= thr / er.FLAT_MARGIN else "free" if m2 <= thr * er.FLAT_MARGIN else "bounded")
        ref = er.restate(np.zeros(T), x, 1.0)
        b = ref.bound[er.K["skew"]]
        assert {"nan": b == 0 and np.isnan(float(ref.values[er.K["skew"]])), "free": b == np.inf,
                "bounded": 0 < b < np.inf}[kind], (kind, b)
        seen.add(kind)
    assert seen == {"nan", "free", "bounded"}


# faults and the case of tests/test_gpu_path_metrics.py that shows each (the same builders, the same seeds)
FAULT_CASES = {
    "chunk_floor": "length_257",
    "peak_from_base": "dd_across_chunks_4149",
    "chunk_peak_restart": "dd_across_chunks_4149",
    "peak_starts_at_one": "dd_shapes_4149",
    "max_four_warps": "length_4149",
    "ddof0": "length_4149",
    "sortino_neg_count": "length_4149",
    "avg_return_zeros": "conditional_513",
    "no_flat_rule": "constant_4149_0.1",
}


@pytest.mark.parametrize("fault", er.FAULTS)
def test_bound_catches_seeded_fault(fault):
    worst, where = 0.0, None
    for r, x, years in _calls(FAULT_CASES[fault]):
        for p in range(len(r)):
            rat = er.ratios(er.kernel_f64(r[p], x[p], years, fault=fault), er.restate(r[p], x[p], years))
            if rat.max() > worst:
                worst, where = float(rat.max()), er.NAMES[int(rat.argmax())]
    REPORT[f"fault {fault}"] = f"{worst:.3g} x bound ({FAULT_CASES[fault]}, {where})"
    assert worst >= 1e3, (fault, worst, where)
