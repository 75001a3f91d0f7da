"""Extended-precision reference, a-priori bounds and a float64 emulation for the Ledoit-Wolf shrinkage stage
(estimators.cu lw_shrink_kernel).

What the stage computes, for one window of K = m = rolling_window - 1 daily excess returns X [m][N] (sklearn's
ledoit_wolf as pypfopt calls it, restated in estimators.cu):
    xbar = t / m (t = X'1),  X_c = X - xbar,  C = X_c'X_c (the Gram stage's centred Gram, input of the stage),
    beta_ = sum_k ||x_k - xbar||^4,  tr = trace C,  fr = ||C||_F^2,
    mu = tr / (m N),  delta_ = fr / m^2,  beta = (beta_/m - delta_) / (N m),  delta = ||C/m - mu I||_F^2 / N,
    s = min(beta, delta) / delta   (sklearn: 0 when min(beta, delta) == 0, and 0 for N = 1),
and hands the solver the system (C + rho I) w = t / (1 - s), rho = s mu m / (1 - s), which is m Sigma_LW w = t with
m Sigma_LW = (1 - s) C + s mu m I scaled by 1 / (1 - s).  A clipped window (s = 1) is solved as mu m I w = t.

Isolating the stage.  The lower off-diagonal of the S1 output is the stage's input C untouched (only the diagonal is
rewritten; a clipped window's is zeroed, and Jorion's S1 of the same batch holds the same bits), so the reference
takes those float64 entries as they are.  It recomputes the diagonal C_ii = sum_k
(x_ki - xbar_i)^2, t and beta_ from X in np.longdouble; the device's C_ii and t are within the Gram stage's
entry-wise bounds B_ii and b_i of these (tests/_gram_ref.py: (K + C_MAT) u times the magnitudes sum_k y_ki^2 +
2 (sum_k y_ki)^2 / K and sum_k y_ki, y = |x| + 2|a|).  delta is evaluated cancellation-free, as
(2 sum_{i>j} C_ij^2 + sum_i (C_ii - tr/N)^2) / (N m^2).  This costs O(m N + N^2) per window at any N, N >= m included.

The bounds (u = 2**-53, a priori, first order).  Every sum the kernel forms is a chain of roundings whose longest
path has n terms: its error is at most n u times the sum of the magnitudes.  The kernel's paths (kernel_depths):
  * r_k = ||x_k - xbar||^2: a lane adds two columns per 64-column step, then 5 shuffle levels: n_r = 2 ceil(N/64) + 5;
  * beta_ = sum_k r_k^2: lane 0 of a warp adds two rows per 16-row step, then block_sum (5 + 5 levels):
    n_b = 2 ceil(K/16) + 11;
  * tr, fr: a thread owns rows i = warp mod 8 and columns j = lane mod 32: n_f = ceil(N/8) ceil(N/32) + 10.
Inputs: xbar = t/m carries e_xbar = b/m + u |xbar|, each centred entry d = x - xbar carries e_d = e_xbar + e_x + u |d|
(e_x: the difference between the rows the kernel reads and the reference's X, 0 for the device's own daily rows;
it also adds sum_k e_x to b and 2 sum_k |d| e_x to B),
so e(r_k) = sum_i 2 |d_ki| e_d,ki + n_r u r_k and e(beta_) = sum_k 2 r_k e(r_k) + n_b u beta_;
e(tr) = sum_i B_ii + n_f u tr and e(fr) = sum_i 2 |C_ii| B_ii + (n_f + 1) u fr (off-diagonal inputs carry no error).
  * mu, beta, delta: the kernel's scalar formulas are then followed operation by operation, each adding its own
    rounding (tests/_solver_ref._Err).  The kernel forms delta as delta_ - 2 mu tr/m + N mu^2: the three terms are each
    up to ~2 delta_ while delta can be far smaller when C/m is close to mu I -- exactly where the intensity clips.  The
    bound therefore scales with delta_ / N (the magnitudes of the terms), not with delta.
  * s: min(. , delta) is 1-Lipschitz, so |ds| <= (e(beta) + e(delta)) / delta + 2u, clipped or not.  N = 1: s = 0.
  * weights.  The kernel uses one rounded value of 1 - s both in rho and in the scale of t, so multiplying its system
    by (1 - s_k) gives (1 - s_k) C_dev + s_k mu_k m I (to the roundings of rho): an error ds in s perturbs the solved
    matrix A = (1 - s) C + s mu m I by about ds ||C||, however close s is to 1 (the relative error of 1 - s itself is not
    amplified into the weights).  Normwise,
        |dA|_2 <= ds |C|_F + max_i B_ii + m (ds mu + e(mu)) + 8 u (s mu m + max_i A_ii),
        |db|_2 <= |b|_2 + 3 u |t|_2,
    eta_in = |dA|_2 / |A|_2 + |db|_2 / |t|_2, and the solver's forward error bound of tests/_chain_ref.solver_bound,
    2 kappa_2(A) (eta_in + 4 sqrt(N) u), holds x = A^-1 t (nu and w1) in the infinity norm; weights = x / gamma add 2u.
  * S1 diagonal and rhs are checked against the kernel's own s_k and mu_k (themselves held to the bounds above):
    S_ii = C_ii + s_k mu_k m / (1 - s_k) to B_ii + 6 u rho + u |S_ii|, rhs = t / (1 - s_k) to (b + 3 u |t|) / (1 - s_k);
    a clipped window has S_ii = fl(mu_k m) exactly, zero off the diagonal and rhs = t to b.
"""
from __future__ import annotations

import numpy as np

from tests import _chain_ref as cr
from tests import _gram_ref as gr
from tests._solver_ref import _Err

U = 2.0 ** -53
LD = np.longdouble
LW_THREADS, LW_WARPS = 256, 8


def _cdiv(a, b):
    return -(-a // b)


def kernel_depths(N: int, K: int):
    """(n_r, n_b, n_f): longest rounding chains of r_k, beta_ and tr / fr in lw_shrink_kernel (module docstring)."""
    return 2 * _cdiv(N, 64) + 5, 2 * _cdiv(K, 16) + 11, _cdiv(N, 8) * _cdiv(N, 32) + 10


def generic_depths(N: int, K: int):
    """Depths that hold for any summation order (sklearn's BLAS products and pairwise sums)."""
    return 0, K + N * N + 1, K + N * N + 1


class LWRef:
    """The stage's reference for one window.  ``X`` [m][N]: the rows the kernel centres (float64); ``S1`` [N][N]: the
    emitted S1 (only its strict lower triangle is read: the kernel's input C); ``a`` [m]: the risk-free adjustments
    (magnitudes of the Gram bounds); ``x_err``: per-entry bound on the difference between the kernel's rows and X."""

    def __init__(self, X, S1, a=None, x_err=0.0, depths=None):
        gr.require_extended_precision()
        X = np.asarray(X, dtype=np.float64)
        K, N = X.shape
        self.K, self.N, self.m = K, N, float(K)
        a = np.zeros(K) if a is None else np.asarray(a, dtype=np.float64)
        y = np.abs(X) + 2.0 * np.abs(a)[:, None]
        ys = y.sum(axis=0)
        self.t_err = (K + gr.C_MAT) * U * ys                                      # b_i
        self.B = (K + gr.C_MAT) * U * ((y * y).sum(axis=0) + 2.0 * ys * ys / K)   # B_ii (centred, den = K)
        Xl = X.astype(LD)
        mL = LD(K)
        self.t = Xl.sum(axis=0)
        xbar = self.t / mL
        D = Xl - xbar
        D2 = D * D
        r = D2.sum(axis=1)
        self.beta_ = (r * r).sum()
        self.Cd = D2.sum(axis=0)
        Lo = np.tril(np.asarray(S1, dtype=np.float64), -1)
        self.C_off = Lo
        off2 = (Lo.astype(LD) ** 2).sum()
        self.tr = self.Cd.sum()
        self.fr = (self.Cd * self.Cd).sum() + 2 * off2
        Nd = LD(N)
        self.mu = self.tr / (mL * Nd)
        self.delta_ = self.fr / (mL * mL)
        self.beta = (self.beta_ / mL - self.delta_) / (Nd * mL)
        self.delta = (2 * off2 + ((self.Cd - self.tr / Nd) ** 2).sum()) / (Nd * mL * mL)
        if N == 1:
            self.s = LD(0)
        else:
            b = min(self.beta, self.delta)
            self.s = LD(0) if b == 0 else b / self.delta
        self.clipped = N > 1 and self.beta >= self.delta

        # ---- error bounds
        n_r, n_b, n_f = depths or kernel_depths(N, K)
        Da = np.abs(D).astype(np.float64)
        xe = np.broadcast_to(np.asarray(x_err, dtype=np.float64), X.shape)
        self.t_err = self.t_err + xe.sum(axis=0)                   # rows the kernel reads differ from X by x_err
        self.B = self.B + 2.0 * (Da * xe).sum(axis=0)
        e_xbar = self.t_err / K + U * np.abs(xbar.astype(np.float64))
        e_d = e_xbar[None, :] + xe + U * Da
        rf = r.astype(np.float64)
        e_r = 2.0 * (Da * e_d).sum(axis=1) + n_r * U * rf
        e_beta_ = float(2.0 * (rf * e_r).sum() + n_b * U * float(self.beta_))
        Cdf = self.Cd.astype(np.float64)
        e_tr = float(self.B.sum() + n_f * U * float(self.tr))
        e_fr = float(2.0 * (np.abs(Cdf) * self.B).sum() + (n_f + 1) * U * float(self.fr))
        tr_, fr_, b_ = _Err(self.tr, e_tr), _Err(self.fr, e_fr), _Err(self.beta_, e_beta_)
        m = self.m
        trace_e = tr_ / m
        mu = trace_e / float(N)
        delta_ = fr_ / (m * m)
        inv = _Err(LD(1) / (Nd * mL), U / (N * m))
        beta = inv * (b_ / m - delta_)
        delta = (delta_ - 2.0 * mu * trace_e + float(N) * mu * mu) / float(N)
        self.e_mu, self.e_beta, self.e_delta = float(mu.e), float(beta.e), float(delta.e)
        if N == 1:
            self.e_s = 0.0
        elif float(self.delta) <= self.e_delta:
            self.e_s = np.inf
        else:
            self.e_s = (self.e_beta + self.e_delta) / float(self.delta) + 2 * U

    # ------------------------------------------------------------------------------------------------- system
    def matrix(self):
        """A = (1 - s) C + s mu m I (longdouble, full), the solved m Sigma_LW."""
        C = self.C_off.astype(LD)
        C = C + C.T
        C[np.diag_indices(self.N)] = self.Cd
        A = (1 - self.s) * C
        A[np.diag_indices(self.N)] += self.s * self.mu * LD(self.m)
        return A, C

    def solution(self):
        """(x = A^-1 t as longdouble, relative infinity-norm bound of the solver's x), or (None, inf) when A is not
        numerically positive definite (m = 2: beta is 0 in exact arithmetic and C has rank 1)."""
        A, C = self.matrix()
        Af = A.astype(np.float64)
        ev = np.linalg.eigvalsh(Af)
        if not ev[0] > 1e3 * U * ev[-1]:
            return None, np.inf
        kappa = float(ev[-1] / ev[0])
        x = cr.refined_solve(A, self.t)
        s, mu, m = float(self.s), float(self.mu), self.m
        Cf = np.linalg.norm(C.astype(np.float64))
        dA = (self.e_s * Cf + float(self.B.max()) + m * (self.e_s * mu + self.e_mu)
              + 8 * U * (s * mu * m + float(np.abs(np.diag(Af)).max())))
        tf = self.t.astype(np.float64)
        eta_in = dA / float(ev[-1]) + (np.linalg.norm(self.t_err) + 3 * U * np.linalg.norm(tf)) / np.linalg.norm(tf)
        return x, cr.solver_bound(self.N, kappa, eta_in)

    def diag_expected(self, s_k: float, mu_k: float):
        """(S1 diagonal the kernel must write given its own s_k and mu_k, entry-wise bound)."""
        m = self.m
        if s_k == 1.0:
            v = np.full(self.N, LD(mu_k) * LD(m))
            return v, U * np.abs(v.astype(np.float64))
        rho = LD(s_k) * LD(mu_k) * LD(m) / (1 - LD(s_k))
        v = self.Cd + rho
        return v, self.B + 6 * U * abs(float(rho)) + U * np.abs(v.astype(np.float64))

    def rhs_expected(self, s_k: float):
        if s_k == 1.0:
            return self.t, self.t_err
        sc = 1 / (1 - LD(s_k))
        return self.t * sc, (self.t_err + 3 * U * np.abs(self.t.astype(np.float64))) * float(sc)


def ratio(got, ref, bound) -> float:
    """max |got - ref| / bound over the entries (inf when an entry is not finite or misses a zero bound)."""
    got = np.asarray(got)
    err = np.abs(got.astype(LD) - np.asarray(ref, dtype=LD)).astype(np.float64)
    bound = np.broadcast_to(np.asarray(bound, dtype=np.float64), err.shape)
    if not np.all(np.isfinite(err)) or np.any((bound == 0) & (err != 0)):
        return np.inf
    with np.errstate(invalid="ignore", divide="ignore"):
        r = np.where(bound > 0, err / bound, 0.0)
    return float(r.max()) if r.size else 0.0


def sklearn_weights(X, gamma: float):
    """(1/gamma) Sigma_LW^-1 mean with sklearn's ledoit_wolf (the annualisation factor cancels)."""
    from sklearn.covariance import ledoit_wolf
    cov, s = ledoit_wolf(X)
    return np.linalg.solve(cov, X.mean(axis=0)) / gamma, float(s)


# ------------------------------------------------------------------------------------------------- emulation
def _xor_tree(v):
    """warp_sum / __shfl_xor_sync tree over the last axis (32 lanes); returns lane 0's value."""
    lanes = np.arange(32)
    for o in (16, 8, 4, 2, 1):
        v = v + v[..., lanes ^ o]
    return v[..., 0]


def _block_sum(v):
    """common.cuh block_sum of 256 thread values [8][32]."""
    w = _xor_tree(np.asarray(v, dtype=np.float64))
    return float(_xor_tree(np.r_[w, np.zeros(32 - LW_WARPS)]))


def emulate(X, t, S1, fixed: bool = True):
    """lw_shrink_kernel in float64, in its summation order (products and sums rounded separately where the kernel
    fuses them: the bound covers both).  X [m][N] the rows, t the device's t, S1 the stage's input C (lower triangle).
    ``fixed=False`` runs the formula without the N = 1 rule and the s = 1 branch.  Returns the scalars, the system's
    full matrix and right-hand side."""
    X = np.asarray(X, dtype=np.float64)
    K, N = X.shape
    m = float(K)
    xbar = np.asarray(t, dtype=np.float64) / m
    J = _cdiv(N, 64)
    Dp = np.zeros((K, 64 * J))
    Dp[:, :N] = X - xbar
    Dp = Dp.reshape(K, J, 32, 2)
    s = np.zeros((K, 32))
    for j in range(J):
        for e in range(2):
            s = s + Dp[:, j, :, e] * Dp[:, j, :, e]
    r = _xor_tree(s)
    b4 = np.zeros((LW_WARPS, 32))
    for w in range(LW_WARPS):
        acc = 0.0
        for k in range(2 * w, K, 2 * LW_WARPS):
            acc = acc + r[k] * r[k]
            if k + 1 < K:
                acc = acc + r[k + 1] * r[k + 1]
        b4[w, 0] = acc
    beta_ = _block_sum(b4)
    S = np.asarray(S1, dtype=np.float64)
    tr = np.zeros((LW_WARPS, 32))
    fr = np.zeros((LW_WARPS, 32))
    for i in range(N):
        w = i % LW_WARPS
        row = np.zeros(_cdiv(i + 1, 32) * 32)
        row[:i + 1] = S[i, :i + 1]
        row = row.reshape(-1, 32)
        for jj in range(row.shape[0]):
            v = row[jj]
            diag = np.arange(32) + 32 * jj == i
            live = np.arange(32) + 32 * jj <= i
            tr[w] = np.where(diag, tr[w] + v, tr[w])
            fr[w] = np.where(live, fr[w] + np.where(diag, v * v, (2.0 * v) * v), fr[w])
    tr, fr = _block_sum(tr), _block_sum(fr)
    Nd = float(N)
    trace_e = tr / m
    mu = trace_e / Nd
    delta_ = fr / (m * m)
    beta = 1.0 / (Nd * m) * (beta_ / m - delta_)
    delta = delta_ - 2.0 * mu * trace_e + Nd * mu * mu
    delta /= Nd
    beta_raw = beta
    beta = min(beta, delta)
    with np.errstate(divide="ignore", invalid="ignore"):
        if fixed:
            shrink = 0.0 if (N == 1 or beta == 0.0) else beta / delta
            clip = shrink == 1.0
            scale = 1.0 if clip else np.float64(1.0) / (1.0 - shrink)
            dg = mu * m if clip else np.float64(shrink) * mu * m / (1.0 - shrink)
        else:
            shrink = 0.0 if beta == 0.0 else beta / delta
            clip = False
            scale = np.float64(1.0) / np.float64(1.0 - shrink)
            dg = np.float64(shrink) * mu * m / np.float64(1.0 - shrink)
    A = np.tril(S, -1)
    A = A + A.T
    if clip:
        A[:] = 0.0
        A[np.diag_indices(N)] = dg
    else:
        A[np.diag_indices(N)] = np.diag(S) + dg
    rhs = scale * np.asarray(t, dtype=np.float64)
    return dict(shrinkage=shrink, mu=mu, beta=beta_raw, delta=delta, scale=scale, diag=dg, A=A, rhs=rhs)


# ------------------------------------------------------------------------------------------------- markets
def iid_returns(K: int, N: int, rng, vol: float = 0.01, drift: float = 3e-4):
    """K i.i.d. equal-volatility daily returns of N assets: the Ledoit-Wolf target mu I is the truth, and the
    intensity clips to 1 in a large share of windows."""
    return rng.standard_normal((K, N)) * vol + drift


def mixed_returns(E, f, c: float):
    """E + c f 1': a common factor of scale c mixed into i.i.d. returns (c = 0 keeps E)."""
    return E + c * f[:, None]


def factor_scale_for(E, f, target: float, lo: float = 0.0, hi: float = 1.0, steps: int = 200):
    """Bisection for the factor scale c at which the reference intensity of E + c f 1' is ``target`` (< 1): s(c)
    falls from 1 (clipped, c = 0) as the common factor grows.  E, f are float64; the returned c is the midpoint of a
    bracket [lo, hi] with s(lo) >= target > s(hi)."""
    def s_of(c):
        X = mixed_returns(E, f, c)
        Xc = X - X.mean(axis=0)
        return LWRef(X, Xc.T @ Xc).s
    while s_of(hi) >= target:
        hi *= 2.0
    for _ in range(steps):
        mid = 0.5 * (lo + hi)
        if mid in (lo, hi):
            break
        if s_of(mid) >= target:
            lo = mid
        else:
            hi = mid
    return 0.5 * (lo + hi)
