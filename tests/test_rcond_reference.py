"""tests/_rcond_ref.py (the definition of the solver's condition estimate) against LAPACK's own dpocon."""
import numpy as np
import pytest
from scipy.linalg.lapack import dpocon

from tests import _rcond_ref as ref

TOL = 1e-14


def _cases():
    rng = np.random.default_rng(20261020)
    out = []
    for k in range(240):
        N = int(rng.integers(2, 121))
        if k % 3 == 0:
            A = ref.gram(N, N + 1, rng)                     # one row above rank deficiency
        elif k % 3 == 1:
            A = ref.gram(N, int(rng.integers(N + 2, 4 * N + 8)), rng)
        else:
            A = ref.spd_with_cond(N, 10.0 ** rng.uniform(0, 12), rng)
        out.append((k, A))
    return out


CASES = _cases()


def _dpocon(L, anorm):
    r, info = dpocon(np.asfortranarray(L), anorm, "L")
    assert info == 0
    return r


@pytest.mark.parametrize("k", range(0, len(CASES), 20))
def test_matches_dpocon_block(k):
    for kk, A in CASES[k:k + 20]:
        L = np.linalg.cholesky(A)
        anorm = ref.anorm1(A)
        got, solves = ref.rcond(L, anorm)
        want = _dpocon(L, anorm)
        assert got > 0.0
        assert abs(got - want) <= TOL * want, f"case {kk}, N={A.shape[0]}: {got!r} vs dpocon {want!r}"
        assert 1 <= solves <= 11


def test_enough_cases():
    assert len(CASES) >= 200
    assert sum(1 for k, A in CASES if k % 3 == 0) >= 50


@pytest.mark.parametrize("N", [1, 2])
def test_tiny(N):
    rng = np.random.default_rng(N)
    for _ in range(20):
        A = ref.spd_with_cond(N, 10.0 ** rng.uniform(0, 8), rng) * rng.uniform(0.1, 10.0)
        L = np.linalg.cholesky(A)
        anorm = ref.anorm1(A)
        got, _ = ref.rcond(L, anorm)
        want = _dpocon(L, anorm)
        assert abs(got - want) <= TOL * want
        if N == 1:
            assert got == pytest.approx(1.0 / (abs(1.0 / A[0, 0]) * anorm), rel=TOL)


def test_anorm_zero():
    L = np.linalg.cholesky(np.eye(4) * 2.0)
    assert ref.rcond(L, 0.0)[0] == 0.0
    assert _dpocon(L, 0.0) == 0.0


def test_anorm1_reads_the_lower_triangle():
    rng = np.random.default_rng(3)
    A = ref.spd_with_cond(7, 100.0, rng)
    S = np.tril(A) + np.triu(rng.standard_normal((7, 7)), 1)     # garbage above the diagonal
    assert ref.anorm1(S) == np.max(np.abs(A).sum(axis=0))


def test_bounds_against_exact_cond():
    """est <= ||A^-1||_1 up to rounding, so rcond >= 1/cond_1; and it is within a factor 10 on these cases."""
    for k, A in CASES[::7]:
        L = np.linalg.cholesky(A)
        r, _ = ref.rcond(L, ref.anorm1(A))
        c1 = np.linalg.cond(A, 1)
        if c1 > 1e10:
            continue
        assert (1 - 1e-6) / c1 <= r <= 10.0 / c1, f"case {k}: rcond {r:.3e}, 1/cond_1 {1 / c1:.3e}"
