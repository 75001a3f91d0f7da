"""CPU tests of the Gram-stage reference (tests/_gram_ref.py): the longdouble sums are exact to far below the bound,
a plain float64 evaluation of the same matrices passes the bound, and every plausible kernel fault -- a row dropped or
doubled, a block boundary off by one row, an overnight return left out, alpha applied twice, the last 128-column tile
lost -- fails it by more than four orders of magnitude."""
from fractions import Fraction

import numpy as np
import pytest

from tests import _gram_ref as gr
from tests._solver_ref import factor_returns

BARS = 78


def _as_fraction(v):
    n, d = np.longdouble(v).as_integer_ratio()
    return Fraction(n, d)


@pytest.fixture(scope="module", autouse=True)
def _extended():
    gr.require_extended_precision()


def _daily(K, N, seed):
    rng = np.random.default_rng(seed)
    X = factor_returns(K, N, rng)
    a = np.full(K, 1.0) * rng.uniform(5e-5, 2e-4, K)
    return X - a[:, None], a


def _intraday(m, N, seed):
    rng = np.random.default_rng(seed)
    return factor_returns(m, N, rng) / np.sqrt(BARS)


@pytest.mark.parametrize("K,N", [(3, 2), (5, 4), (9, 3)])
def test_longdouble_reference_matches_exact_sums(K, N):
    X, a = _daily(K, N, 10 + K)
    H = _intraday(K + 2, N, 20 + K)
    alpha = 37.25
    T, t = gr.daily_ref(X, a)
    S0 = gr.s0_ref(H, alpha)
    J = gr.centred_ref(T, t, K + 1)
    G, g = gr.fraction_gram(X)
    Gh, gh = gr.fraction_gram(H)
    m = H.shape[0]
    tol = 4 * K * 2.0 ** -64           # a K-term longdouble sum, relative to its magnitude
    for i in range(N):
        assert abs(_as_fraction(t.value[i]) - g[i]) <= Fraction(tol) * Fraction(float(t.A[i]))
        for j in range(N):
            A = Fraction(float(T.A[i, j]))
            assert abs(_as_fraction(T.value[i, j]) - G[i][j]) <= Fraction(tol) * A
            s0 = Fraction(alpha) * (Gh[i][j] - gh[i] * gh[j] / m)
            assert abs(_as_fraction(S0.value[i, j]) - s0) <= Fraction(4 * (m + 4) * 2.0 ** -64) * Fraction(float(S0.A[i, j]))
            jx = G[i][j] - g[i] * g[j] / (K + 1)
            assert abs(_as_fraction(J.value[i, j]) - jx) <= Fraction(4 * (K + 4) * 2.0 ** -64) * Fraction(float(J.A[i, j]))


# ------------------------------------------------------------------------------------------------- mutations
N_MUT = 130        # two 128-column tiles: the last one holds columns 128 and 129


def _case(name):
    if name == "hf20k":
        H = _intraday(20_000, N_MUT, 3)
        alpha = 252.0 * 20_000 / 19_999
        return "S0", H, None, gr.s0_ref(H, alpha), alpha
    K = int(name[1:])
    X, a = _daily(K, N_MUT, K)
    T, _ = gr.daily_ref(X, a)
    return "T", X, a, T, 1.0


CASES = ["K33", "K251", "hf20k"]


@pytest.fixture(scope="module")
def cases():
    return {name: _case(name) for name in CASES}


def _mutate(kind, rows, ref, alpha, mutation):
    """A faulty kernel's result, as a rank-one change (or a scaling) of the correct matrix."""
    V = ref.value.copy()
    Y = rows.astype(np.longdouble)
    n = rows.shape[0]
    mid = n // 2
    s = np.longdouble(alpha)
    if mutation == "row_dropped":
        V -= s * np.outer(Y[mid], Y[mid])
    elif mutation == "row_doubled":
        V += s * np.outer(Y[mid], Y[mid])
    elif mutation == "block_boundary_shifted":           # the row at a block edge lands in neither block, the next one in both
        e = n // 3
        V += s * (np.outer(Y[e + 1], Y[e + 1]) - np.outer(Y[e], Y[e]))
    elif mutation == "overnight_rank1_left_out":         # the first return of a day (the gathered overnight row)
        k = (n // BARS // 2) * BARS if n >= 2 * BARS else 0
        V -= s * np.outer(Y[k], Y[k])
    elif mutation == "alpha_twice":
        V *= np.longdouble(alpha if kind == "S0" else 2.0)
    elif mutation == "last_tile_column_zeroed":
        V[:, 128:] = 0
    return V


@pytest.mark.parametrize("name", CASES)
def test_float64_evaluation_passes_the_bound(cases, name):
    kind, rows, a, ref, alpha = cases[name]
    if kind == "T":
        got = rows.T @ rows
    else:
        m = rows.shape[0]
        g = rows.sum(axis=0)
        got = alpha * (rows.T @ rows - np.outer(g, g) / m)
    r = gr.lower_ratio(got, ref)
    assert r < 1.0, r


MUTATIONS = ["row_dropped", "row_doubled", "block_boundary_shifted", "overnight_rank1_left_out", "alpha_twice",
             "last_tile_column_zeroed"]


@pytest.mark.parametrize("mutation", MUTATIONS)
@pytest.mark.parametrize("name", CASES)
def test_checker_flags_mutation(cases, name, mutation):
    """Each fault exceeds the bound by > 1e4: the check would still fail with its bound loosened ten thousand times."""
    kind, rows, a, ref, alpha = cases[name]
    bad = _mutate(kind, rows, ref, alpha, mutation)
    assert gr.lower_ratio(bad.astype(np.float64), ref) > 1e4
    loose = gr.Ref(ref.value, ref.A * 1e4, ref.K)
    assert gr.lower_ratio(bad.astype(np.float64), loose) > 1.0


def test_column_subset_and_vectors():
    """A column-subset reference equals the same columns of the full one; the moment vectors follow S0 and t."""
    rng = np.random.default_rng(7)
    X, a = _daily(40, 300, 8)
    cols = gr.edge_columns(300, rng)
    assert {0, 1, 126, 127, 128, 129, 254, 255, 256, 257, 298, 299} <= set(cols.tolist())
    T, t = gr.daily_ref(X, a)
    Ts, _ = gr.daily_ref(X, a, cols)
    assert np.array_equal(Ts.value, T.value[:, cols])
    assert np.allclose(Ts.A, T.A[:, cols], rtol=1e-13, atol=0)        # float64 magnitudes: BLAS blocking may differ
    H = _intraday(200, 300, 9)
    S0 = gr.s0_ref(H, 50.0)
    w0 = rng.uniform(0.5, 1.5, 300)
    w0 /= w0.sum()
    s0w0, v0, (c, c_err), (rhs, rhs_err) = gr.moments_ref(S0, t, w0, 60.0)
    got = (S0.value.astype(np.float64) @ w0)
    assert gr.lower_ratio(got, s0w0, gr.C_VEC) < 1.0
    assert gr.lower_ratio(got * (1 + 1e-9), s0w0, gr.C_VEC) > 1.0
    cf = float(c)
    assert gr.scalar_ratio(cf, c, c_err) < 1.0
    assert gr.scalar_ratio(cf * (1 + 1e-10), c, c_err) > 1.0
    r = cf * got + t.value.astype(np.float64)
    assert np.max(np.abs(r - rhs.astype(np.float64)) / rhs_err) < 1.0
