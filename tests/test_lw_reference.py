"""The Ledoit-Wolf stage's reference (tests/_lw_ref.py) on the CPU: against the installed sklearn, one feature and
clipped windows included, and a float64 emulation of lw_shrink_kernel held to the stage's a-priori bounds.  The
emulation also shows why a clipped window needs its own branch: 1 / (1 - s) is inf at s = 1."""
import numpy as np
import pytest

from tests import _lw_ref as lr

GAMMA = 3.0
CASES = {                                     # name: (N, K, kind)
    "one asset": (1, 50, "iid"),
    "two assets": (2, 17, "factor"),
    "iid N=20 (clips)": (20, 120, "iid"),
    "N=33 K=16": (33, 16, "factor"),
    "N=64 > m=32": (64, 32, "iid"),
    "factor N=65 K=251": (65, 251, "factor"),
}


def _returns(N, K, kind, rng):
    if kind == "iid":
        return lr.iid_returns(K, N, rng)
    from tests._solver_ref import factor_returns
    return factor_returns(K, N, rng)


def _windows(name, n=12):
    N, K, kind = CASES[name]
    rng = np.random.default_rng(sum(map(ord, name)))
    for _ in range(n):
        X = _returns(N, K, kind, rng)
        Xc = X - X.mean(axis=0)
        yield X, Xc.T @ Xc


@pytest.fixture(scope="module", autouse=True)
def _extended():
    lr.gr.require_extended_precision()


@pytest.mark.parametrize("name", list(CASES))
def test_reference_matches_sklearn(name):
    """Shrinkage and weights of sklearn.covariance.ledoit_wolf, held to the reference's bounds with depths that hold
    for any summation order; one asset gives shrinkage 0 and clipped windows exactly 1 in both."""
    N, K, _ = CASES[name]
    clipped = 0
    for X, C in _windows(name):
        ref = lr.LWRef(X, C, depths=lr.generic_depths(N, K))
        w_sk, s_sk = lr.sklearn_weights(X, GAMMA)
        if N == 1:
            assert s_sk == 0.0 and ref.s == 0
        else:
            assert abs(s_sk - float(ref.s)) <= ref.e_s, (s_sk, float(ref.s), ref.e_s)
        if ref.clipped:
            clipped += 1
            assert s_sk == 1.0
        x, eps = ref.solution()
        xf = x.astype(np.float64) / GAMMA
        assert np.max(np.abs(w_sk - xf)) <= eps * np.max(np.abs(xf))
    if name.startswith("iid N=20"):
        assert clipped >= 4                    # i.i.d. equal-volatility windows clip often


@pytest.mark.parametrize("name", list(CASES))
def test_kernel_emulation_within_bound(name):
    """The kernel's scalar block, its S1 diagonal, rhs and solution, emulated in float64 in the kernel's summation
    order, against the reference and its kernel-depth bounds."""
    for X, C in _windows(name):
        ref = lr.LWRef(X, C)
        em = lr.emulate(X, X.sum(axis=0), C)
        assert lr.ratio(em["mu"], ref.mu, ref.e_mu) < 1
        assert lr.ratio(em["beta"], ref.beta, ref.e_beta) < 1
        assert lr.ratio(em["delta"], ref.delta, ref.e_delta) < 1
        assert lr.ratio(em["shrinkage"], ref.s, ref.e_s) < 1
        d, d_err = ref.diag_expected(em["shrinkage"], em["mu"])
        assert lr.ratio(np.diag(em["A"]), d, d_err) < 1
        rhs, rhs_err = ref.rhs_expected(em["shrinkage"])
        assert lr.ratio(em["rhs"], rhs, rhs_err) < 1
        x, eps = ref.solution()
        xe = np.linalg.solve(em["A"], em["rhs"])
        assert np.max(np.abs(xe - x.astype(np.float64))) <= eps * float(np.max(np.abs(x)))


def test_clipped_window_needs_its_own_system():
    """At s = 1 the general formula's scale 1 / (1 - s) and rho are inf and the solve gives NaN weights; the
    clipped system mu m I w = t gives sklearn's weights, mean / (gamma mu)."""
    seen = 0
    for X, C in _windows("iid N=20 (clips)", n=30):
        ref = lr.LWRef(X, C)
        if not ref.clipped:
            continue
        seen += 1
        old = lr.emulate(X, X.sum(axis=0), C, fixed=False)
        assert old["shrinkage"] == 1.0 and np.isinf(old["scale"]) and np.isinf(old["diag"])
        assert np.all(np.isinf(np.diag(old["A"]))) and np.all(np.isinf(old["rhs"][old["rhs"] != 0]))
        with np.errstate(invalid="ignore"):                 # the first forward-substitution step: inf / inf
            assert np.isnan(old["rhs"][0] / np.sqrt(old["A"][0, 0]))
        new = lr.emulate(X, X.sum(axis=0), C)
        assert new["shrinkage"] == 1.0 and new["scale"] == 1.0
        assert np.array_equal(new["A"], np.diag(np.full(X.shape[1], new["mu"] * X.shape[0])))
        assert np.array_equal(new["rhs"], X.sum(axis=0))
        w = np.linalg.solve(new["A"], new["rhs"]) / GAMMA
        w_sk, s_sk = lr.sklearn_weights(X, GAMMA)
        x, eps = ref.solution()
        assert s_sk == 1.0
        assert np.max(np.abs(w - w_sk)) <= 2 * eps * np.max(np.abs(w_sk))
        mean_over_mu = X.mean(axis=0) / (GAMMA * float(ref.mu))
        assert np.max(np.abs(w - mean_over_mu)) <= eps * np.max(np.abs(mean_over_mu))
    assert seen >= 8


def test_one_asset_rounded_delta():
    """One asset: delta is 0 in exact arithmetic, but the kernel's rounded delta is not in many windows; without
    sklearn's one-feature rule min(beta, delta) / delta is then 1 (or worse), with the rule it is always 0."""
    rng = np.random.default_rng(3)
    nonzero = 0
    for _ in range(300):
        X = lr.iid_returns(60, 1, rng)
        Xc = X - X.mean(axis=0)
        C = Xc.T @ Xc
        old = lr.emulate(X, X.sum(axis=0), C, fixed=False)
        new = lr.emulate(X, X.sum(axis=0), C)
        assert new["shrinkage"] == 0.0 and new["scale"] == 1.0 and new["diag"] == 0.0
        if old["delta"] != 0.0:
            nonzero += 1
            assert old["shrinkage"] != 0.0
    assert nonzero >= 30


@pytest.mark.parametrize("log2_gap", [20, 40])
def test_near_clipped_windows(log2_gap):
    """s = 1 - 2^-k, built by mixing a common factor into i.i.d. returns: the emulated kernel's weights stay within a
    bound that does not grow with 1 / (1 - s)."""
    rng = np.random.default_rng(log2_gap)
    E = lr.iid_returns(120, 20, rng)
    f = rng.standard_normal(120) * 0.01
    while lr.LWRef(E, (E - E.mean(0)).T @ (E - E.mean(0))).s < 1:       # start from a clipped window
        E = lr.iid_returns(120, 20, rng)
    target = 1.0 - 2.0 ** -log2_gap
    X = lr.mixed_returns(E, f, lr.factor_scale_for(E, f, target))
    Xc = X - X.mean(axis=0)
    C = Xc.T @ Xc
    ref = lr.LWRef(X, C)
    assert abs(float(1 - ref.s) / 2.0 ** -log2_gap - 1.0) < 1e-3
    em = lr.emulate(X, X.sum(axis=0), C)
    assert em["shrinkage"] < 1.0
    assert lr.ratio(em["shrinkage"], ref.s, ref.e_s) < 1
    x, eps = ref.solution()
    assert eps < 1e-9
    xe = np.linalg.solve(em["A"], em["rhs"])
    assert np.max(np.abs(xe - x.astype(np.float64))) <= eps * float(np.max(np.abs(x)))
