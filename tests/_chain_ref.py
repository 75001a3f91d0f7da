"""Extended-precision reference, a-priori bound and a float64 emulation for the Jeffreys / Jorion chain
(jeffreys_chain.cu): windows of consecutive trade dates solved relative to a factorised base window.

What the chain computes, for window w = b + k of a group with base b (k = 1 .. G-1):
    x = J_w^-1 t_w  (Jeffreys: J_w = T_w - t_w t_w'/n;  Jorion: C_w = T_w - t_w t_w'/(n-1), and also C_w^-1 1)
by the Woodbury identity J_w = J_b + U C U' with U = [k new rows | k old rows | p_w - p_b | 1 | t_w | t_b] and
C^-1 = diag(+I, -I, -[0 1; 1 0], -n, +n) (Jorion: n - 1 in place of n), a system of m = 2k + 4 unknowns.

The reference.  J_w and t_w are evaluated in np.longdouble (64-bit mantissa) from the daily log returns l and the
risk-free adjustments a of the window's K = n - 1 rows (tests/_gram_ref.py: T = X'X with x = l - a 1, t = X'1).  The
raw Gram of consecutive windows slides by one row added and one removed, also in longdouble, so a batch costs one
N x K x N product however many windows it has; each slide adds 2 2**-64 of the magnitudes, 2**9 times below the
bound over a few hundred slides.  x_ref solves the longdouble J_w with float64 Cholesky and three refinement steps
whose residuals are taken in longdouble (error about kappa 5e-20).

The bound (u = 2**-53, a priori, not tuned).  The chain's result is the exact solution of a perturbed problem:
  * the inputs.  J_b is the device's Gram, within the entry-wise bound B_b of tests/_gram_ref.py; the columns of U are
    the device's log returns, p and t, within the same kind of bound, so J_b + U C U' is within B_w (the entry-wise
    bound of J_w) of J_w, and t_w within its own bound.  Normwise, eta_in = max(|B_b|_2 / |J_b|_2, |B_w|_2 / |J_w|_2)
    + |b_t|_2 / |t_w|_2, and the perturbation bound of a linear system gives 2 kappa_2(J_w) eta_in (the factor 2
    covers 1 / (1 - kappa eta) while kappa eta <= 1/2).
  * the arithmetic.  The substitutions against the base factor have the solver's backward error 4 sqrt(N) u relative
    to J_b, so Y = J_b^-1 U and y_t carry kappa_2(J_b) times that; the m x m elimination and the update x = y_t - Y c
    add m-term sums (2m u) and O(1) roundings (8 u).  Relative to J_w these act through both kappas, hence
        2 (kappa_2(J_b) + kappa_2(J_w)) (4 sqrt(N) + 2m + 8) u.
So
    |x - x_ref|_inf / |x_ref|_inf <= eps = 2 kappa_2(J_w) eta_in + 2 (kappa_2(J_b) + kappa_2(J_w)) (4 sqrt(N) + 2m + 8) u.
Woodbury is not backward stable in general (the capacitance matrix can be far worse conditioned than J_w), so this
is a claim the tests check, not a theorem; the rank guard of the planner (chain only when n - 1 >= N + 2G + 8) keeps
the capacitance system away from the rank limit, and the tests run exactly at that margin.  Weights and nu are x / gamma
and x (one more rounding); v1 = x't carries |x - x_ref|_inf |t|_1 + |x_ref|' b_t + (N + 2) u |x_ref|'|t|.  For the
per-window solver (base windows) the same argument gives 2 kappa_2(J) (eta_in + 4 sqrt(N) u).

Singular windows.  A window whose own matrix is exactly singular gives a capacitance system that is singular only in
exact arithmetic; its smallest Gauss-Jordan pivot is then some 1e-19 of max |M| or less, while regular windows keep
pivots above 1e-9 of max |M|.  The kernel flags a window whose pivot falls to TAU max |M| or below (TAU = 2**-40).
"""
from __future__ import annotations

import numpy as np
import scipy.linalg as sla

from tests import _gram_ref as gr
from tests import _solver_ref as sr

U = 2.0 ** -53
LD = np.longdouble
TAU = 2.0 ** -40
COL_NEW, COL_OLD, COL_PD, COL_ONE, COL_T, COL_T0 = 0, 7, 14, 21, 22, 29


# ------------------------------------------------------------------------------------------------- references
def log_returns(prices: np.ndarray) -> np.ndarray:
    """Row r = log(P_r / P_r-1) (row 0 is NaN): the daily log returns the library computes."""
    out = np.full(prices.shape, np.nan)
    out[1:] = np.log(prices[1:] / prices[:-1])
    return out


class WindowRefs:
    """J_w (or Jorion's C_w) and t_w of a batch's windows, as tests/_gram_ref.Ref, with the raw Gram slid in longdouble
    between consecutive windows.  ``lr`` are the daily log returns (log_returns), ``rf_row`` the risk-free rate per
    daily row, ``batch`` the planned WindowBatch."""

    def __init__(self, lr: np.ndarray, rf_row: np.ndarray, batch, jorion: bool = False):
        self.lr, self.rf_row, self.batch = lr, rf_row, batch
        self.n = int(batch.rolling_window)
        self.den = self.n - 1 if jorion else self.n
        self._rows = None
        self._G = None

    def _gram(self, rows):
        if self._rows is not None and len(rows) == len(self._rows) and rows[0] == self._rows[0] + 1:
            old, new = self.lr[self._rows[0]].astype(LD), self.lr[rows[-1]].astype(LD)
            self._G = self._G + np.outer(new, new) - np.outer(old, old)
        elif self._rows is None or not np.array_equal(rows, self._rows):
            L = self.lr[rows].astype(LD)
            self._G = L.T @ L
        self._rows = rows
        return self._G

    def __call__(self, i: int):
        """(J, t) of window i: Ref objects in longdouble with their entry-wise bounds."""
        rows = gr.daily_return_rows(int(self.batch.day_row[i]), self.n)
        a = gr.daily_adjustments(self.rf_row, rows, int(self.batch.span_days[i]))
        G = self._gram(rows)
        L = self.lr[rows]
        Ll, al = L.astype(LD), a.astype(LD)
        p = Ll.T @ al
        s = Ll.sum(axis=0)
        T = G - p[:, None] - p[None, :] + al @ al
        t = s - al.sum()
        y = np.abs(L - a[:, None]) + 2.0 * np.abs(a)[:, None]
        K = len(rows)
        Tr = gr.Ref(T, y.T @ y, K)
        tr = gr.Ref(t, y.sum(axis=0), K)
        return gr.centred_ref(Tr, tr, self.den), tr


def eta(ref: gr.Ref) -> float:
    """Normwise relative bound |B|_2 / |value|_2 of a Ref (B >= 0 entry-wise, so |E|_2 <= |B|_2)."""
    B = ref.bound()
    v = np.asarray(ref.value, dtype=np.float64)
    if B.ndim == 1:
        return float(np.linalg.norm(B) / np.linalg.norm(v))
    return float(np.abs(np.linalg.eigvalsh(B)).max() / np.abs(np.linalg.eigvalsh(v)).max())


def kappa2(J) -> float:
    ev = np.linalg.eigvalsh(np.asarray(J, dtype=np.float64))
    return float(ev[-1] / ev[0]) if ev[0] > 0 else np.inf


def chain_bound(N: int, k: int, kappa_b: float, kappa_w: float, eta_in: float) -> float:
    m = 2 * k + 4
    return 2.0 * kappa_w * eta_in + 2.0 * (kappa_b + kappa_w) * (4.0 * np.sqrt(N) + 2 * m + 8) * U


def solver_bound(N: int, kappa: float, eta_in: float) -> float:
    return 2.0 * kappa * (eta_in + 4.0 * np.sqrt(N) * U)


def refined_solve(J, b) -> np.ndarray:
    """x = J^-1 b for a longdouble J (and b) to about kappa 5e-20, as np.longdouble."""
    return sr.refined_solve(np.asarray(J, dtype=LD), np.asarray(b, dtype=LD))


def v1_bound(x_ref, eps: float, t: gr.Ref) -> float:
    xa = np.abs(np.asarray(x_ref, dtype=np.float64))
    ta = np.abs(np.asarray(t.value, dtype=np.float64))
    N = len(xa)
    return float(eps * xa.max() * ta.sum() + xa @ t.bound() + (N + 2) * U * (xa @ ta))


# ------------------------------------------------------------------------------------------------- emulation
def c_inverse(k: int, beta_den: float):
    """C^-1 of window b + k in the kernel's row order: +1 (new rows), -1 (old rows), -[0 1; 1 0] (p_w - p_b, 1),
    -n (t_w), +n (t_b); Jorion uses n - 1.  Returns the m x m matrix."""
    m = 2 * k + 4
    C = np.zeros((m, m))
    C[np.arange(k), np.arange(k)] = 1.0
    C[np.arange(k, 2 * k), np.arange(k, 2 * k)] = -1.0
    C[2 * k, 2 * k + 1] = C[2 * k + 1, 2 * k] = -1.0
    C[2 * k + 2, 2 * k + 2] = -beta_den
    C[2 * k + 3, 2 * k + 3] = beta_den
    return C


def col_of(a: int, k: int) -> int:
    if a < k:
        return COL_NEW + a
    if a < 2 * k:
        return COL_OLD + (a - k)
    if a == 2 * k:
        return COL_PD + (k - 1)
    if a == 2 * k + 1:
        return COL_ONE
    if a == 2 * k + 2:
        return COL_T + (k - 1)
    return COL_T0


def gauss_jordan(M: np.ndarray, R: np.ndarray):
    """The kernel's elimination: for each column s, the not yet used row with the largest |M[:, s]| (ties to the lower
    row) eliminates column s from every other row (Gauss-Jordan).  Returns (solution [m][r], smallest pivot / max |M|)."""
    m = M.shape[0]
    A = np.concatenate([M, R], axis=1).astype(np.float64)
    scale = np.abs(M).max()
    used = np.zeros(m, dtype=bool)
    piv_row = np.empty(m, dtype=int)
    rel = np.inf
    for s in range(m):
        cand = np.where(used, -1.0, np.abs(A[:, s]))
        bl = int(np.argmax(cand))            # first maximum: the lowest row among ties
        rel = min(rel, cand[bl] / scale)
        pv = A[bl, s]
        for r in range(m):
            if r != bl:
                f = A[r, s] / pv
                A[r, s + 1:] = A[r, s + 1:] - f * A[bl, s + 1:]
                A[r, s] = 0.0
        used[bl] = True
        piv_row[s] = bl
    with np.errstate(divide="ignore", invalid="ignore"):
        sol = np.stack([A[piv_row[s], m:] / A[piv_row[s], s] for s in range(m)])
    return sol, rel


def emulate_group(Lfac: np.ndarray, lr: np.ndarray, pvec: np.ndarray, t: np.ndarray, day_b: int, n: int, nb: int,
                  beta_den: float):
    """The chain of one group in float64: Lfac the base's Cholesky factor, lr the daily log returns by row, pvec[k] and
    t[k] the vectors p and t of window b + k (k = 0 .. nb).  Returns for k = 1 .. nb a dict with x = J^-1 t_w and
    the smallest relative pivot."""
    N = Lfac.shape[0]
    Rb = np.zeros((N, 32))
    for c in range(nb):
        Rb[:, COL_NEW + c] = lr[day_b + 1 + c]
        Rb[:, COL_OLD + c] = lr[day_b - n + 2 + c]
        Rb[:, COL_PD + c] = pvec[1 + c] - pvec[0]
        Rb[:, COL_T + c] = t[1 + c]
    Rb[:, COL_ONE] = 1.0
    Rb[:, COL_T0] = t[0]
    Z = sla.solve_triangular(Lfac, Rb, lower=True)
    Wm = Z.T @ Z
    Y = sla.solve_triangular(Lfac, Z, lower=True, trans="T")
    out = []
    for k in range(1, nb + 1):
        cols = [col_of(a, k) for a in range(2 * k + 4)]
        tcol = COL_T + (k - 1)
        M = Wm[np.ix_(cols, cols)] + c_inverse(k, beta_den)
        c, rel = gauss_jordan(M, Wm[cols, tcol][:, None])
        out.append(dict(x=Y[:, tcol] - Y[:, cols] @ c[:, 0], rel_pivot=rel))
    return out


# ------------------------------------------------------------------------------------------------- markets
def jeffreys_spec(N: int, n: int, strategy: str = "jeffreys"):
    return dict(weighting_strategy=strategy, size=N, risk_aversion=3, turnover_cost=15, rebalancing_frequency="daily",
                rolling_window=n, rolling_window_frequency="daily", mcm_scaling=None, display_name="x")


def chain_market(N: int, n: int, W: int, seed: int, rf_zero: bool = False):
    """A seeded market with W consecutive rebalance dates of rolling window n at its end.  Returns (mkt, d_idx)."""
    from incorporating_different_sources_b200.synthetic import generate_market
    D = n + W + 3
    mkt = generate_market(N, D, seed=seed, bars_per_day=2)
    if rf_zero:
        mkt.rf[:] = 0.0
    return mkt, list(range(D - W, D))


def flatten(mkt, asset: int, lo: int, hi: int):
    """Asset ``asset`` has zero log return on daily return rows [lo, hi) (its price is constant on rows lo-1 .. hi-1)
    and the returns it had before from row hi on."""
    P = mkt.prices
    old = P[hi - 1, asset]
    P[lo:hi, asset] = P[lo - 1, asset]
    P[hi:, asset] *= P[hi - 1, asset] / old


def rf_rows(mkt) -> np.ndarray:
    from incorporating_different_sources_b200.windows import ffill_rows
    return ffill_rows(mkt.dates, mkt.dates, mkt.rf)


def plan(mkt, spec, d_idx):
    from incorporating_different_sources_b200.windows import plan_daily_windows
    return plan_daily_windows(spec, mkt.dates, d_idx, need_hf=False)
