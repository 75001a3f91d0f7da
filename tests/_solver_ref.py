"""Matrix generators and a high-precision reference for the Cholesky solver tests.

The reference solves S x = b with LAPACK (scipy's cho_factor / cho_solve) and refines x three times with residuals
b - S x evaluated in np.longdouble (80-bit extended precision on x86-64, 64-bit mantissa).  Its error is about
kappa * 5e-20, three orders of magnitude below every bound the GPU solver is held to.

Bounds (u = 2**-53, a priori, not tuned):
  * normwise backward error  eta = |b - S x|_inf / (|S|_inf |x|_inf + |b|_inf) <= 4 sqrt(N) u;
  * forward error            |x - x_ref|_inf / |x_ref|_inf <= 2 kappa_2 * 4 sqrt(N) u  (the perturbation bound
    2 kappa eta / (1 - kappa eta) for a backward error eta in S and b).
Everything is seeded: a child process regenerates the same problems from the same seed.
"""
from __future__ import annotations

import numpy as np
import scipy.linalg as sla

U = 2.0 ** -53
LD = np.longdouble


def require_extended_precision():
    if np.finfo(LD).nmant < 63:
        raise RuntimeError("np.longdouble is not 80-bit extended precision on this platform: the reference needs it")


def eta_bound(N: int) -> float:
    return 4.0 * np.sqrt(N) * U


def forward_bound(N: int, kappa: float) -> float:
    return 2.0 * kappa * eta_bound(N)


def symmetric_from_lower(S: np.ndarray) -> np.ndarray:
    """The matrix the solver sees: the lower triangle of S, mirrored."""
    L = np.tril(S)
    return L + np.tril(S, -1).T


def refined_solve(S: np.ndarray, b: np.ndarray, steps: int = 3) -> np.ndarray:
    """x = S^-1 b (S symmetric positive definite, float64 or np.longdouble; b [N] or [N][k]) to about kappa * 5e-20, as
    np.longdouble.  The residuals are taken with S as given (a longdouble S is factorised rounded to float64)."""
    require_extended_precision()
    cf = sla.cho_factor(np.asarray(S, dtype=np.float64), lower=True, check_finite=True)
    S_ld = np.asarray(S, dtype=LD)
    b_ld = np.asarray(b, dtype=LD)
    x = sla.cho_solve(cf, np.asarray(b, dtype=np.float64)).astype(LD)
    for _ in range(steps):
        r = b_ld - S_ld @ x
        x = x + sla.cho_solve(cf, r.astype(np.float64)).astype(LD)
    return x


def backward_error(S: np.ndarray, x: np.ndarray, b: np.ndarray) -> float:
    """Normwise backward error in the infinity norm, evaluated in extended precision."""
    S_ld = S.astype(LD)
    x_ld = np.asarray(x, dtype=LD)
    b_ld = np.asarray(b, dtype=LD)
    r = b_ld - S_ld @ x_ld
    den = np.max(np.sum(np.abs(S_ld), axis=1)) * np.max(np.abs(x_ld)) + np.max(np.abs(b_ld))
    return float(np.max(np.abs(r)) / den)


def forward_error(x: np.ndarray, x_ref: np.ndarray) -> float:
    x_ref = np.asarray(x_ref, dtype=LD)
    return float(np.max(np.abs(np.asarray(x, dtype=LD) - x_ref)) / np.max(np.abs(x_ref)))


def kappa2(S: np.ndarray) -> float:
    ev = np.linalg.eigvalsh(S)
    return float(ev[-1] / ev[0])


# ---------------------------------------------------------------------------------------------------- generators
def spd_with_kappa(N: int, kappa: float, rng: np.random.Generator) -> np.ndarray:
    """S = Q diag(lambda) Q' with lambda log-spaced from 1 down to 1/kappa, symmetrised; the problem is this float64
    matrix (its kappa_2 is kappa to a few parts in kappa * 1e-16)."""
    if N == 1:
        return np.array([[1.0]])
    Q, R = np.linalg.qr(rng.standard_normal((N, N)))
    Q *= np.sign(np.diag(R))
    lam = np.logspace(0.0, -np.log10(kappa), N)
    S = (Q * lam) @ Q.T
    return 0.5 * (S + S.T)


def factor_returns(m: int, N: int, rng: np.random.Generator, k: int = 3) -> np.ndarray:
    """m daily returns of N assets from a k-factor model (market-like first factor, idiosyncratic noise)."""
    F = rng.standard_normal((m, k)) * np.array([0.01] + [0.005] * (k - 1))[:k]
    B = rng.standard_normal((N, k)) * 0.5 + np.r_[1.0, np.zeros(k - 1)]
    E = rng.standard_normal((m, N)) * rng.uniform(0.005, 0.02, N)
    return F @ B.T + E + 3e-4


def project_like(N: int, rng: np.random.Generator):
    """The Jeffreys matrix of the project: J = X'X - t t'/n of n - 1 = N + 10 factor-model returns; rhs t."""
    n = N + 11
    X = factor_returns(n - 1, N, rng)
    t = X.sum(axis=0)
    J = X.T @ X - np.outer(t, t) / n
    return 0.5 * (J + J.T), t


def badly_scaled(S: np.ndarray, rng: np.random.Generator):
    """D S D with D log-spaced over 1e-4 .. 1e4 (shuffled); returns (D S D, D)."""
    N = S.shape[0]
    d = np.logspace(-4.0, 4.0, N)
    rng.shuffle(d)
    A = (S * d[:, None]) * d[None, :]
    return 0.5 * (A + A.T), d


def equilibrate(S: np.ndarray):
    """H = D^-1 S D^-1 with D = sqrt(diag S): Cholesky's accuracy depends on kappa_2(H), not on kappa_2(S)."""
    d = np.sqrt(np.diag(S))
    return (S / d[:, None]) / d[None, :], d


def failing_pivot_matrix(N: int, ks, rng: np.random.Generator) -> np.ndarray:
    """S = L diag(d) L' with unit lower-triangular L (small off-diagonal entries) and d_k = -1 at every k of ks, else
    d in [0.5, 2]: the first non-positive pivot of S is at min(ks), clear of rounding."""
    L = np.eye(N) + np.tril(rng.standard_normal((N, N)), -1) * (0.3 / np.sqrt(N))
    d = rng.uniform(0.5, 2.0, N)
    for k in ks:
        d[k] = -1.0
    S = (L * d) @ L.T
    return 0.5 * (S + S.T)


def healthy_matrix(N: int, rng: np.random.Generator) -> np.ndarray:
    return failing_pivot_matrix(N, [], rng)


def pivot_columns(N: int):
    return sorted({k for k in (0, 1, 7, 8, 31, 32, 33, 64, 95, N - 2, N - 1) if 0 <= k < N})


def two_failures(N: int):
    """Two failing columns in panels owned by different cluster ranks (panels of 32 columns: consecutive panels are
    owned by consecutive ranks), or None when N has a single panel."""
    if N <= 32:
        return None
    if N <= 64:
        return 5, N - 1
    return 33, min(N - 1, 70)


# ---------------------------------------------------------------------------------------------------- Jorion
class _Err:
    """A value with a first-order bound on its absolute error: each operation adds its own float64 rounding."""

    def __init__(self, v, e):
        self.v = np.asarray(v, dtype=LD)
        self.e = np.asarray(e, dtype=LD)

    def _wrap(self, o):
        return o if isinstance(o, _Err) else _Err(o, 0)

    def __add__(self, o):
        o = self._wrap(o)
        v = self.v + o.v
        return _Err(v, self.e + o.e + U * np.abs(v))

    __radd__ = __add__

    def __sub__(self, o):
        o = self._wrap(o)
        v = self.v - o.v
        return _Err(v, self.e + o.e + U * np.abs(v))

    def __rsub__(self, o):
        return self._wrap(o) - self

    def __mul__(self, o):
        o = self._wrap(o)
        v = self.v * o.v
        return _Err(v, self.e * np.abs(o.v) + o.e * np.abs(self.v) + self.e * o.e + U * np.abs(v))

    __rmul__ = __mul__

    def __truediv__(self, o):
        o = self._wrap(o)
        v = self.v / o.v
        rel_o = o.e / np.abs(o.v)
        return _Err(v, (self.e / np.abs(o.v) + np.abs(v) * rel_o) / (1 - rel_o) + U * np.abs(v))

    def __rtruediv__(self, o):
        return self._wrap(o) / self

    def sum(self, weights=None):
        w = np.ones_like(self.v) if weights is None else np.asarray(weights, dtype=LD)
        v = np.sum(w * self.v)
        n = self.v.size
        return _Err(v, np.sum(np.abs(w) * self.e) + n * U * np.sum(np.abs(w * self.v)))


def jorion_reference(C: np.ndarray, t: np.ndarray, m: int, risk_aversion: float, kappa: float, eps: float = None):
    """Jorion's Bayes-Stein portfolio (oracle.bayes_oracle.jorion_window, portfolio_calculations.py:851-895) restated
    on the centred Gram C = (m-1) V_hat, t = m mu_hat and m, evaluated on the refined y = C^-1 t and z = C^-1 1.
    Returns values and first-order error bounds: y and z carry the forward-error bound, every later operation its
    own float64 rounding, as the solver's epilogue evaluates it.  ``eps`` replaces the solver's forward-error bound of
    y and z (relative, infinity norm) where another stage produced them (the chain of tests/_chain_ref.py)."""
    N = C.shape[0]
    yz = refined_solve(C, np.stack([np.asarray(t, dtype=LD), np.ones(N, dtype=LD)], axis=1))
    eps = forward_bound(N, kappa) if eps is None else eps
    y = _Err(yz[:, 0], eps * np.max(np.abs(yz[:, 0])))
    z = _Err(yz[:, 1], eps * np.max(np.abs(yz[:, 1])))
    md, Nd = float(m), float(N)
    kap = md / ((md - Nd - 2.0) * (md - 1.0))                 # V_bar = kap C (:876-879)
    sy, sz, ty = y.sum(), z.sum(), y.sum(weights=t)
    one_vinv_one = sz / kap
    mu_g = (sy / md) / sz                                     # :882
    q = (ty / (md * md) - (sy / md) * (sy / md) / sz) / kap   # (mu_hat - mu_g 1)' V_bar^-1 (mu_hat - mu_g 1)
    lam = (Nd + 2.0) / q                                      # :885
    v = (Nd + 2.0) / ((Nd + 2.0) + md * q)                    # :887
    a = 1.0 + 1.0 / (md + lam)                                # V_PJ = a V_bar + b 11' (:888)
    b = lam / (md * (md + 1.0 + lam)) / one_vinv_one
    # nu = V_PJ^-1 mu_PJ, mu_PJ = (1 - v) mu_hat + v mu_g 1 (:889), by Sherman-Morrison
    r = ((1.0 - v) / md) * y / (a * kap) + (v * mu_g) * z / (a * kap)
    s = z / (a * kap)
    nu = r - s * (b * r.sum() / (1.0 + b * s.sum()))
    w = nu * (1.0 / risk_aversion)
    return dict(weights=w, nu=nu, y=y, mu_g=mu_g, lambda_hat=lam, v_hat=v, q=q, one_vinv_one=one_vinv_one)


def jorion_problem(N: int, rng: np.random.Generator):
    """Centred Gram C of m = 2N + 10 factor-model returns, t = sum of the returns, m."""
    m = 2 * N + 10
    X = factor_returns(m, N, rng)
    t = X.sum(axis=0)
    Xc = X - t / m
    C = Xc.T @ Xc
    return 0.5 * (C + C.T), t, m
