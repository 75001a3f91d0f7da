"""CPU tests of the solver tests' reference and generators (tests/_solver_ref.py): the refined solve is far more
accurate than the bounds the GPU solver is held to, LAPACK itself meets a quarter of the backward-error bound on
the sweep's matrices, and the failing-pivot constructions fail exactly where LAPACK's dpotrf says."""
import numpy as np
import pytest
import scipy.linalg as sla
import scipy.linalg.lapack as lapack

from tests import _solver_ref as ref


def _mp_solve(S, b, dps=40):
    mpmath = pytest.importorskip("mpmath")
    with mpmath.workdps(dps):
        x = mpmath.lu_solve(mpmath.matrix(S.tolist()), mpmath.matrix(b.tolist()))
        return np.array([float(x[i]) for i in range(len(b))], dtype=np.float64), x


def test_longdouble_is_extended_precision():
    ref.require_extended_precision()


@pytest.mark.parametrize("N", [5, 17, 33])
@pytest.mark.parametrize("kappa", [1e2, 1e10])
def test_reference_against_mpmath(N, kappa):
    mpmath = pytest.importorskip("mpmath")
    rng = np.random.default_rng(1000 + N)
    S = ref.spd_with_kappa(N, kappa, rng)
    b = rng.standard_normal(N)
    x = ref.refined_solve(S, b)
    _, x_mp = _mp_solve(S, b)
    with mpmath.workdps(40):
        num = max(abs(mpmath.mpf(str(x[i])) - x_mp[i]) for i in range(N))
        den = max(abs(x_mp[i]) for i in range(N))
        err = float(num / den)
    # the GPU forward-error bound at this N and kappa; the reference must sit 1000x inside it
    assert err <= ref.forward_bound(N, kappa) / 1000, (err, ref.forward_bound(N, kappa))


SWEEP_NS = [1, 2, 7, 8, 9, 15, 16, 17, 31, 32, 33, 63, 64, 65, 96, 127, 128, 129, 255, 257, 500, 511, 512, 513]


@pytest.mark.parametrize("N", SWEEP_NS)
def test_lapack_meets_quarter_of_the_backward_bound(N):
    rng = np.random.default_rng(2000 + N)
    mats = [ref.spd_with_kappa(N, k, rng) for k in (1e2, 1e8, 1e12)]
    if N >= 2:
        J, _ = ref.project_like(N, rng)
        mats.append(J)
        mats.append(ref.badly_scaled(mats[0], rng)[0])
    for S in mats:
        b = rng.standard_normal(N)
        x = sla.cho_solve(sla.cho_factor(S, lower=True), b)
        assert ref.backward_error(S, x, b) <= 0.25 * ref.eta_bound(N)


@pytest.mark.parametrize("N", [8, 33, 100, 257, 500])
def test_failing_pivot_constructions_match_dpotrf(N):
    rng = np.random.default_rng(3000 + N)
    cases = [[k] for k in ref.pivot_columns(N)]
    two = ref.two_failures(N)
    if two:
        cases.append(list(two))
    for ks in cases:
        S = ref.failing_pivot_matrix(N, ks, rng)
        _, info = lapack.dpotrf(S, lower=1, clean=0)
        assert info == min(ks) + 1, (ks, info)
    # NaN at (k, k): OpenBLAS's dpotrf does not test pivots for NaN, so pin the construction instead: the leading
    # k x k block factors, so the first pivot that is not positive is the NaN at column k
    for k in ref.pivot_columns(N):
        S = ref.healthy_matrix(N, rng)
        assert lapack.dpotrf(S, lower=1)[1] == 0
        S[k, k] = np.nan
        assert k == 0 or lapack.dpotrf(S[:k, :k], lower=1)[1] == 0
        assert np.isnan(S[k, k])


def test_healthy_matrices_factor():
    rng = np.random.default_rng(4)
    for N in (8, 33, 100, 257, 500):
        assert lapack.dpotrf(ref.healthy_matrix(N, rng), lower=1)[1] == 0


def test_jorion_reference_matches_the_oracle_formulas():
    """The Sherman-Morrison restatement on (C, t, m) equals the explicit-inverse form of
    oracle.bayes_oracle.jorion_window on the returns."""
    rng = np.random.default_rng(5)
    N = 31
    m = 2 * N + 10
    X = ref.factor_returns(m, N, rng)
    t = X.sum(axis=0)
    Xc = X - t / m
    C = Xc.T @ Xc
    got = ref.jorion_reference(0.5 * (C + C.T), t, m, 3.0, ref.kappa2(C))
    # the oracle's own arithmetic (jorion_window) on the same returns
    mu_hat = X.mean(axis=0)
    V_bar = m / (m - N - 2) * np.cov(X, rowvar=False)
    Vi = np.linalg.inv(V_bar)
    one = np.ones(N)
    ovo = one @ Vi @ one
    mu_g = one @ Vi @ mu_hat / ovo
    diff = mu_hat - mu_g * one
    q = diff @ Vi @ diff
    lam = (N + 2) / q
    v = (N + 2) / ((N + 2) + m * q)
    V_PJ = (1 + 1 / (m + lam)) * V_bar + lam / (m * (m + 1 + lam)) * np.outer(one, one) / ovo
    w = 1 / 3.0 * np.linalg.solve(V_PJ, (1 - v) * mu_hat + v * mu_g * one)
    np.testing.assert_allclose(np.asarray(got["weights"].v, dtype=float), w, rtol=1e-9)
    for k, val in (("mu_g", mu_g), ("q", q), ("lambda_hat", lam), ("v_hat", v), ("one_vinv_one", ovo)):
        assert abs(float(got[k].v) - val) <= 1e-9 * abs(val), k
