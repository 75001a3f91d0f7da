"""Extended-precision reference and a-priori entry-wise bound for the Gram stage (gram_dmma.cu and its feeders).

What each output is (oracle/bayes_oracle.py, include/bayes_portfolio.h), for one window:
  * X [K][N]: the window's daily excess log returns (K = rolling_window - 1 rows, x_k = l_k - a_k 1 with l_k the log
    return and a_k the frequency-adjusted risk-free rate, :31-62).  T = X'X, t = X'1 (:180-182, :222).
  * H [m][N]: the window's KEPT intraday log returns (the rows dropna keeps, tests/_dropna_ref.py).
    S0 = alpha (H'H - m hbar hbar'), hbar = H'1 / m, alpha = n0 m / (m - 1)   (n0 cov(H) m, :314-333).
  * S1 = S0 + T (:358);  J = T - t t'/n with n = rolling_window (:600-601);  Jorion's centred C = T - t t'/(n - 1).
  * rhs = c S0 w0 + t (:489), v0 = w0'S0 w0, c = 2 n0 / (k + sqrt(k^2 + 4 n0 v0)), k = n0 + N + 2 (:415-418).
Sums are evaluated in np.longdouble (64-bit mantissa): a K-term sum then carries at most K 2**-64 of its magnitude,
2**11 times below the bound below.

The bound (u = 2**-53, a priori, not tuned).  Every route of the library -- from scratch, block tiles added from a
store, range / run sums, pre-summed scans, chunks -- forms the same products and only associates their sum
differently; any summation tree over K terms is within gamma_K = K u / (1 - K u) of the exact sum, times the sum of
the magnitudes.  So for one entry

    |E_ij| <= (K + c) u A_ij

with K the number of rows summed and A_ij the sum of the magnitudes of everything the kernels add:
  * T: the kernel contracts the raw log returns l and subtracts the rank-2 risk-free terms p_i + p_j of the epilogue
    (pvec, themselves K-term sums of a_k l_ki and a_k^2).  With y_ki = |x_ki| + 2|a_k| >= |l_ki| + |a_k| every one
    of those terms is bounded by A_ij = sum_k y_ki y_kj.  t: A_i = sum_k y_ki.
  * S0: alpha (sum_k |h_ki h_kj| + 2 s_i s_j / m), s_i = sum_k |h_ki|.  The mean term m hbar_i hbar_j is at most
    s_i s_j / m; each hbar carries gamma_m of s / m, so its product carries twice that: hence the factor 2.
  * S1: A(S0) + A(T), K = max(m, K).  J / C: A(T) + 2 A_i A_j / n (resp. n - 1), by the same argument as S0.
The constant c collects the O(1) roundings outside the sums:
    1  gamma_K versus K u (K u < 3e-12 here),
    4  reference inputs: the rows are the device's (daily) or np.log(P_r / P_r-1) of the same correctly rounded ratio
       (intraday), one ulp of log apart on each of the two factors of a product (2 + 2),
    2  the excess-return row x = fl(l - a) that the reference reads versus the l and a the kernel reads (one per factor),
    3  the epilogue's three subtractions (- p_i - p_j - beta g_i g_j), each rounding a partial result bounded by A,
    2  beta g_i g_j (two products), 1 alpha times the sum, 1 S0 + T in S1,
    = 14, rounded up to C_MAT = 16.
Vectors and scalars that contract a matrix with w0 (S0 w0, v0, rhs) add N terms per level: (K + N + C_VEC) u with
the magnitudes contracted the same way (C_VEC = 2 C_MAT covers the two levels' O(1) terms and c's rounding).
"""
from __future__ import annotations

from fractions import Fraction

import numpy as np

U = 2.0 ** -53
LD = np.longdouble
C_MAT = 16
C_VEC = 2 * C_MAT


def require_extended_precision():
    if np.finfo(LD).nmant < 63:
        raise RuntimeError("np.longdouble is not 80-bit extended precision on this platform: the reference needs it")


def _cols(N, cols):
    return np.arange(N) if cols is None else np.asarray(cols)


# ------------------------------------------------------------------------------------------------- window inputs
def daily_adjustments(rf_row: np.ndarray, rows: np.ndarray, span_days: int) -> np.ndarray:
    """a_k = (1 + rf)^(span / K / 365) - 1 at the window's return rows (:40-48): float64, used for magnitudes only."""
    K = len(rows)
    return (1.0 + rf_row[rows]) ** (float(span_days) / K / 365.0) - 1.0


def daily_return_rows(day_row: int, rolling_window: int) -> np.ndarray:
    """Daily rows of the window's K = rolling_window - 1 returns (return row r is l(P_r / P_r-1))."""
    return np.arange(day_row - rolling_window + 2, day_row + 1)


def intraday_rows(hf_prices: np.ndarray, lo: int, hi: int) -> np.ndarray:
    """The kept intraday log returns of price rows [lo, hi): float64 [m][N] (dropna of :314)."""
    h = np.log(hf_prices[lo + 1:hi] / hf_prices[lo:hi - 1])
    return h[~np.isnan(h).any(axis=1)]


# ------------------------------------------------------------------------------------------------- references
class Ref:
    """A reference matrix (or vector) in longdouble, its magnitude A and the number of summed rows K.  Matrices may be
    column subsets: ``value`` and ``A`` are then [N][len(cols)] and ``cols`` names the columns."""

    def __init__(self, value, A, K, cols=None):
        self.value = np.asarray(value, dtype=LD)
        self.A = np.asarray(A, dtype=np.float64)
        self.K = int(K)
        self.cols = cols

    def bound(self, c=C_MAT):
        return (self.K + c) * U * self.A


def daily_ref(X: np.ndarray, a: np.ndarray, cols=None):
    """(T, t) of the rows X [K][N] (float64, the device's excess returns) with risk-free adjustments a [K]."""
    K, N = X.shape
    cs = _cols(N, cols)
    Xl = X.astype(LD)
    y = np.abs(X) + 2.0 * np.abs(a)[:, None]
    T = Ref(Xl.T @ Xl[:, cs], y.T @ y[:, cs], K, cols)
    t = Ref(Xl.sum(axis=0), y.sum(axis=0), K)
    return T, t


def s0_ref(H: np.ndarray, alpha: float, cols=None):
    """S0 = alpha (H'H - m hbar hbar') of the kept intraday rows H [m][N]; also returns (g = H'1, s = sum |h|)."""
    m, N = H.shape
    cs = _cols(N, cols)
    Hl = H.astype(LD)
    g = Hl.sum(axis=0)
    al = LD(alpha)
    S0 = al * (Hl.T @ Hl[:, cs] - np.outer(g, g[cs]) / LD(m))
    s = np.abs(H).sum(axis=0)
    A = abs(alpha) * (np.abs(H).T @ np.abs(H[:, cs]) + 2.0 * np.outer(s, s[cs]) / m)
    return Ref(S0, A, m, cols)


def sum_ref(P: Ref, Q: Ref):
    """S1 = S0 + T."""
    return Ref(P.value + Q.value, P.A + Q.A, max(P.K, Q.K), P.cols)


def centred_ref(T: Ref, t: Ref, den: int):
    """T - t t'/den: J (den = rolling_window) or Jorion's C (den = rolling_window - 1)."""
    cs = _cols(T.value.shape[0], T.cols)
    v = T.value - np.outer(t.value, t.value[cs]) / LD(den)
    return Ref(v, T.A + 2.0 * np.outer(t.A, t.A[cs]) / den, T.K, T.cols)


def moments_ref(S0: Ref, t: Ref, w0: np.ndarray, n0: float):
    """(S0 w0, v0, c, rhs) as Refs (S0 must be complete, not a column subset); the bound of c follows from the bound
    of v0: dc/dv0 = -c^2 / sqrt(k^2 + 4 n0 v0)."""
    assert S0.cols is None
    N = S0.value.shape[0]
    wl = np.asarray(w0, dtype=LD)
    aw = np.abs(w0)
    K = S0.K + N
    s0w0 = Ref(S0.value @ wl, S0.A @ aw, K)
    v0 = Ref(wl @ S0.value @ wl, aw @ S0.A @ aw, K + N)
    k = LD(n0) + LD(N) + LD(2)
    sq = np.sqrt(k * k + LD(4) * LD(n0) * v0.value)
    c = LD(2) * LD(n0) / (k + sq)
    dv0 = float(v0.bound(C_VEC))
    c_err = float(c * c / sq) * dv0 + 8 * U * float(c)
    rhs = c * s0w0.value + t.value
    rhs_err = float(c) * s0w0.bound(C_VEC) + c_err * np.abs(s0w0.value.astype(np.float64)) + t.bound() \
        + 2 * U * np.abs(rhs.astype(np.float64))
    return s0w0, v0, (c, c_err), (rhs, rhs_err)


# ------------------------------------------------------------------------------------------------- checking
def lower_ratio(got: np.ndarray, ref: Ref, c=C_MAT) -> float:
    """max over the checked entries of |got - ref| / bound: over the lower triangle of a full matrix, over every row of
    a column subset, over every entry of a vector.  < 1 passes.  Entries whose bound is 0 must match exactly."""
    got = np.asarray(got)
    if ref.cols is not None:
        got = got[:, ref.cols]
        keep = np.ones(got.shape, dtype=bool)
    elif got.ndim == 2:
        keep = np.tril(np.ones(got.shape, dtype=bool))
    else:
        keep = np.ones(got.shape, dtype=bool)
    err = np.abs(got.astype(LD) - ref.value).astype(np.float64)[keep]
    bnd = ref.bound(c)[keep]
    if np.any((bnd == 0) & (err != 0)):
        return np.inf
    if not np.all(np.isfinite(err)):
        return np.inf
    with np.errstate(invalid="ignore", divide="ignore"):
        r = np.where(bnd > 0, err / bnd, 0.0)
    return float(r.max()) if r.size else 0.0


def scalar_ratio(got: float, value, err: float) -> float:
    e = abs(float(LD(got) - LD(value)))
    return e / err if err > 0 else (0.0 if e == 0 else np.inf)


def edge_columns(N: int, rng: np.random.Generator, n_random: int = 16) -> np.ndarray:
    """Columns checked when N is too large for a full longdouble product: the tile edges and 16 seeded random ones."""
    edge = {0, 1, 126, 127, 128, 129, 254, 255, 256, 257, N - 2, N - 1}
    rand = rng.choice(N, size=min(n_random, N), replace=False)
    return np.array(sorted({int(c) for c in edge | set(rand.tolist()) if 0 <= c < N}))


# ------------------------------------------------------------------------------------------------- exact sums
def fraction_gram(Y: np.ndarray):
    """Exact Y'Y and Y'1 of a small float64 matrix, as Fractions."""
    K, N = Y.shape
    F = [[Fraction(float(v)) for v in row] for row in Y]
    G = [[sum((F[k][i] * F[k][j] for k in range(K)), Fraction(0)) for j in range(N)] for i in range(N)]
    g = [sum((F[k][i] for k in range(K)), Fraction(0)) for i in range(N)]
    return G, g
