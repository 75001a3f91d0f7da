"""LAPACK's dpocon / dlacn2 restated in NumPy: the definition of the solver's condition estimate (BP_SCAL_RCOND).

``rcond(L, anorm)`` is the reciprocal 1-norm condition estimate of A = L L' from its lower Cholesky factor L, exactly as
``dpocon`` computes it: ``est`` = dlacn2's Hager-Higham estimate of ||A^-1||_1 (ITMAX = 5, sign rule x >= 0 -> +1,
idamax = the first index of the largest |x_i|), with A^-1 v applied as two triangular solves with L, and rcond =
(1 / est) / anorm.  Edge rules as in LAPACK: anorm == 0 gives 0, N == 1 gives 1 / (|A^-1| anorm), and a solve whose
1-norm is not finite gives 0 (dpocon's exit when the scaled solve would overflow).

``solves_used`` counts the applications of A^-1 in dpocon's order (the GPU kernel merges the last one into the first).
"""
from __future__ import annotations

import numpy as np
from scipy.linalg import solve_triangular

ITMAX = 5


def anorm1(S: np.ndarray) -> float:
    """max_j sum_i |A_ij| of the symmetric A whose lower triangle is that of S."""
    A = np.tril(S) + np.tril(S, -1).T
    return float(np.max(np.sum(np.abs(A), axis=0))) if A.size else 0.0


def _apply_inv(L: np.ndarray, v: np.ndarray) -> np.ndarray:
    y = solve_triangular(L, v, lower=True, check_finite=False)
    return solve_triangular(L, y, lower=True, trans="T", check_finite=False)


def _signs(x: np.ndarray) -> np.ndarray:
    return np.where(x >= 0.0, 1.0, -1.0)


def inv_norm1_estimate(L: np.ndarray):
    """dlacn2's estimate of ||(L L')^-1||_1; returns (est, solves), est = 0 after a non-finite solve."""
    N = L.shape[0]
    solves = 0

    def apply(v):
        nonlocal solves
        solves += 1
        x = _apply_inv(L, v)
        return x, float(np.sum(np.abs(x)))

    x, est = apply(np.full(N, 1.0 / N))
    if not np.isfinite(est):
        return 0.0, solves
    if N == 1:
        return est, solves
    isgn = _signs(x)
    x, s = apply(isgn)
    if not np.isfinite(s):
        return 0.0, solves
    j = int(np.argmax(np.abs(x)))
    it = 2
    while True:
        e = np.zeros(N)
        e[j] = 1.0
        x, s = apply(e)
        if not np.isfinite(s):
            return 0.0, solves
        estold, est = est, s
        if np.array_equal(_signs(x), isgn) or est <= estold:      # repeated sign vector, or cycling
            break
        isgn = _signs(x)
        x, s = apply(isgn)
        if not np.isfinite(s):
            return 0.0, solves
        jlast, j = j, int(np.argmax(np.abs(x)))
        if x[jlast] != abs(x[j]) and it < ITMAX:
            it += 1
            continue
        break
    i = np.arange(N, dtype=np.float64)
    alt = np.where(np.arange(N) % 2 == 0, 1.0, -1.0) * (1.0 + i / (N - 1))
    x, s = apply(alt)
    if not np.isfinite(s):
        return 0.0, solves
    temp = 2.0 * (s / (3.0 * N))
    return max(est, temp), solves


def rcond(L: np.ndarray, anorm: float):
    """dpocon(L', anorm) for the lower Cholesky factor L: returns (rcond, solves)."""
    if L.shape[0] == 0:
        return 1.0, 0
    if anorm == 0.0:
        return 0.0, 0
    est, solves = inv_norm1_estimate(np.asarray(L, dtype=np.float64))
    return ((1.0 / est) / anorm if est != 0.0 else 0.0), solves


def spd_with_cond(N: int, cond2: float, rng: np.random.Generator) -> np.ndarray:
    """Q diag(logspace(0, -log10 cond2)) Q' with a random orthogonal Q: 2-norm condition number cond2."""
    Q, _ = np.linalg.qr(rng.standard_normal((N, N)))
    d = np.logspace(0.0, -np.log10(cond2), N) if N > 1 else np.ones(1)
    A = (Q * d) @ Q.T
    return (A + A.T) / 2


def gram(N: int, m: int, rng: np.random.Generator) -> np.ndarray:
    """Sample Gram of m centred rows: m = N + 1 is one row above rank deficiency (a Jeffreys window with n - 1 = N + 1)."""
    X = rng.standard_normal((m, N)) * rng.uniform(0.5, 2.0, N)
    X -= X.mean(axis=0)
    return X.T @ X
