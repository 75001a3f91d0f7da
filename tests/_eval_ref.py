"""Extended-precision restatement, a-priori bound and a float64 emulation of the path-metrics stage
(eval_kernels.cu path_metrics_kernel, reached through bp_path_metrics / evaluation.path_metrics).

What the kernel computes for one series of n = T simple returns r and excess returns x (oracle/eval_oracle.path_row,
the QuantStats formulas as restated there), with e = 1 / years formed in float64 as both the kernel and the oracle form
it, and the wealth curve W_k = prod_{i <= k} (1 + r_i), k = 0 .. T - 1 (its first point is W_0 = 1 + r_0, not 1):
    Cum. Return = W_{T-1} - 1,  CAGR = |W_{T-1}|^e - 1,  Max. DD = min_k W_k / max_{j <= k} W_j - 1,
    Calmar = CAGR / |Max. DD|,  Avg. Loss / Return / Win = mean of the r < 0 / r != 0 / r > 0 (NaN when none),
    Best / Worst Day = max / min r,  Ann. Vol. = sd(r) sqrt(252),  Daily VaR = mean(r) - z sd(r) (z = 1.6448536269514729),
    Sharpe = mean(x) / sd(x) sqrt(252),  sharpe_per_period = mean(x) / sd(x),  sd with ddof = 1,
    Sortino = mean(x) / sqrt(sum_{x < 0} x^2 / n) sqrt(252),
    skew = m3 / m2^1.5,  kurtosis = m4 / m2^2,  m_k = sum (x - mean)^k / n,
and skew / kurtosis are NaN for a flat sample, by scipy.stats' rule m2 <= (eps mean)^2 (eps = 2**-52).  A division by
zero gives +-inf, or NaN for 0 / 0, as the oracle's NumPy division does.

:func:`restate` evaluates the statistics with the arithmetic of a chosen number type: ``np.longdouble`` for the
reference (64-bit mantissa, 2**11 below the bound), or ``fractions.Fraction`` with sqrt and pow from mpmath at 256
bits (EXACT), to show at small T that the longdouble evaluation is itself accurate.

The bound (u = 2**-53, a priori from the inputs, not tuned to measured errors; c = C_EV = 16 absorbs the O(1)
roundings outside the sums).  All quantities below are the exact ones.
  * Sums.  Any summation tree over n terms returns the exact sum plus at most gamma_n = n u / (1 - n u) times the sum
    of the magnitudes; zeros add exactly and counts (integers < 2**53) are exact.  Means: e_r = (T + c) u sum |r| / n,
    likewise e_x; Avg. Loss / Return / Win over k terms: (k + c) u sum |r_i| / k.
  * Wealth points.  The kernel's W_k is 1 + r_i rounded k + 1 times and multiplied with k rounded products, whether it
    comes from a chunk product, the combine's base * cmax or the second pass's running product: its relative error is
    at most w = (2T + c) u.  Hence Cum. Return: w |W| + 2u |cum| (the final subtraction rounds by up to u |cum|, which
    alone nearly reaches u when the wealth is close to 0); CAGR: pow turns the relative error w into e w and adds at
    most 2 ulp, so W^e (e w + 3u) + 2u |CAGR|.  Each ratio W_k / peak_k carries 2w + u relative, the minimum of
    perturbed ratios is off by at most the largest perturbation and |ratio| <= 1, so Max. DD: 2w + 2u + u |DD|.
    Calmar: (E_cagr + |Calmar| E_dd) / (|DD| - E_dd) + 2u |Calmar|.
  * Central moments.  A deviation b_i = fl(x_i - mean') with mean' = mean + d, |d| <= e_x.  Since sum (x_i - mean) = 0,
    d enters the second moment at second order only: |x2' - M2| <= (T + c) u M2 + 2 n e_x^2 (M2 = n m2).  The sd
    sqrt(M2 / (n - 1)) then errs by min(sqrt(E2 / (n - 1)), E2 / (2 sqrt(M2 (n - 1)))) + 2u sd, which stays finite
    for a constant series (M2 = 0).
  * Sharpe, Sortino, volatility, VaR.  mean / sd errs by (|mean| E_sd + sd e_x) / (sd (sd - E_sd)): the factor
    |mean| / sd is the condition number, and e_x / sd is the same factor times (T + c) u.  Sortino's downside
    D = sqrt(sum_{x<0} x^2 / n) has no mean in it: relative error (T + c) u / 2 + 2u.  VaR: e_r + z E_sd + 2u |VaR|.
    A series with sd = 0 and mean != 0 has Sharpe = +-inf; the kernel's mean error may stand in for a spread, so its
    value is only held to the sign and to |Sharpe| >= (|mean| - e_x) / E_sd (``lo``).
  * Skewness and kurtosis.  The same expansion with the third and fourth absolute moments as magnitudes:
        E3 = 3 e_x M2 + n e_x^3 + (T + c) u sum (|b| + e_x)^3,
        E4 = 4 e_x |sum b^3| + 6 e_x^2 M2 + n e_x^4 + (T + c) u sum (|b| + e_x)^4,
    and with rho = E2 / M2 <= 0.1, E_skew = E3 / n / m2^1.5 (1 + 2 rho) + |skew| (2 rho + 6u),
    E_kurt = E4 / n / m2^2 (1 + 3 rho) + kurt (3 rho + 6u).  Beyond rho = 0.1 there is no claim.
  * The flat rule.  NaN whenever the exact m2 is 0, and whenever m2 <= (eps mean)^2 / 10**3; finite and held to the
    bound when m2 > 10**3 (eps mean)^2.  In between the kernel's summation order and the exact one may disagree: no
    claim (FLAT_MARGIN).
  * Exact outputs.  Best and Worst Day involve no arithmetic.  A non-decreasing curve has Max. DD = 0.0 exactly: every
    factor 1 + r rounds to >= 1, so each running product is >= the last, the combine's base * cmax of a chunk is the
    next chunk's base, and every ratio is 1.  A -100 % day gives W = 0 from there on: Cum. Return, CAGR and Max. DD
    are exactly -1.  +-inf and NaN from a zero downside, sd or drawdown sit where the reference has them.

:func:`kernel_f64` evaluates the kernel's float64 arithmetic in its order (per-thread strided partials, the xor
butterfly of block_sum, the chunked scan of the wealth curve and thread 0's combine), or in another summation order
and chunk count to show the bound holds for any order, optionally with one seeded fault (FAULTS).
"""
from __future__ import annotations

from dataclasses import dataclass
from fractions import Fraction
from itertools import accumulate
from operator import mul

import numpy as np

from tests._loop_ref import kernel_sum

U = 2.0 ** -53
EPS = 2.0 ** -52
LD = np.longdouble
C_EV = 16
Z95 = 1.6448536269514729
FLAT_MARGIN = 1e3
THREADS = 256
NAMES = ("Cum. Return", "CAGR", "Sharpe", "Sortino", "Max. DD", "Calmar", "Avg. Loss", "Avg. Return", "Avg. Win",
         "Best Day", "Worst Day", "Ann. Vol.", "Daily VaR", "skew", "kurtosis", "sharpe_per_period")
K = {name: i for i, name in enumerate(NAMES)}
FAULTS = ("chunk_floor", "peak_from_base", "chunk_peak_restart", "peak_starts_at_one", "max_four_warps", "ddof0",
          "sortino_neg_count", "avg_return_zeros", "no_flat_rule")


def require_extended_precision():
    if np.finfo(LD).nmant < 63:
        raise RuntimeError("np.longdouble is not 80-bit extended precision on this platform: the reference needs it")


@dataclass
class EvalRef:
    """Reference statistics of one series (number type of the evaluation) and, for the longdouble run, their bounds:
    0 = bit-exact (or the same NaN / +-inf), inf = no claim; ``lo`` > 0 on a +-inf reference = the kernel may return a
    finite value of the same sign and at least this magnitude."""
    values: np.ndarray
    bound: np.ndarray = None
    lo: np.ndarray = None


# ------------------------------------------------------------------------------------------------- number types
class _LD:
    @staticmethod
    def cv(v):
        return np.asarray(v, dtype=np.float64).astype(LD)

    @staticmethod
    def total(v):
        return np.sum(v, dtype=LD) if len(v) else LD(0)

    @staticmethod
    def sqrt(v):
        return np.sqrt(LD(v))

    @staticmethod
    def pow(a, e):
        return LD(a) ** LD(e)

    @staticmethod
    def cumprod(v):
        return np.cumprod(v, dtype=LD)

    const = staticmethod(LD)


class _Exact:
    """Fractions; sqrt and pow rounded from mpmath at 256 bits."""
    PREC = 256

    @staticmethod
    def cv(v):
        return np.array([Fraction(float(a)) for a in np.ravel(v)], dtype=object)

    @staticmethod
    def total(v):
        return sum(list(v), Fraction(0))

    @staticmethod
    def _mp(f):
        import mpmath
        return mpmath.mpf(f.numerator) / f.denominator

    @staticmethod
    def _frac(m):
        man, exp = m.man_exp
        return Fraction(int(man)) * Fraction(2) ** int(exp)

    def sqrt(self, v):
        import mpmath
        with mpmath.workprec(self.PREC):
            return self._frac(mpmath.sqrt(self._mp(Fraction(v))))

    def pow(self, a, e):
        import mpmath
        with mpmath.workprec(self.PREC):
            return self._frac(mpmath.power(self._mp(Fraction(a)), self._mp(Fraction(e))))

    @staticmethod
    def cumprod(v):
        return np.array(list(accumulate(v, mul)), dtype=object)

    const = staticmethod(Fraction)


LONGDOUBLE = _LD()
EXACT = _Exact()


def _div(a, b):
    """a / b with the IEEE result of a division by zero (the oracle's NumPy division)."""
    if b == 0:
        return float("nan") if a == 0 else float(np.copysign(np.inf, float(a)))
    return a / b


# ------------------------------------------------------------------------------------------------- restatement
def restate(r, x, years, A=LONGDOUBLE) -> EvalRef:
    """The 16 statistics of one series in the arithmetic of ``A``; with LONGDOUBLE also their bounds."""
    r64, x64 = np.asarray(r, dtype=np.float64), np.asarray(x, dtype=np.float64)
    T = len(r64)
    e = 1.0 / float(years)
    R, X = A.cv(r64), A.cv(x64)
    one, n = A.const(1), A.const(T)
    sq252 = A.sqrt(A.const(252))
    W = A.cumprod(one + R)
    if A is LONGDOUBLE:
        mdd = np.min(W / np.maximum.accumulate(W)) - one
    else:
        mdd = min(w / p for w, p in zip(W, accumulate(W, max))) - one
    total = W[-1]
    cagr = A.pow(abs(total), e) - one
    # the mean of a constant series is that constant (a longdouble sum of its copies need not be exact)
    mr = R[0] if np.all(r64 == r64[0]) else A.total(R) / n
    mx = X[0] if np.all(x64 == x64[0]) else A.total(X) / n
    a, b = R - mr, X - mx
    M2r, M2x = A.total(a * a), A.total(b * b)
    S3, S4 = A.total(b * b * b), A.total(b * b * b * b)
    sd_r, sd_x = A.sqrt(M2r / (n - one)), A.sqrt(M2x / (n - one))
    dn2 = A.total(X[x64 < 0] * X[x64 < 0])
    down = A.sqrt(dn2 / n)
    nan = float("nan")
    cnt = {k: int(np.count_nonzero(m)) for k, m in (("neg", r64 < 0), ("nz", r64 != 0), ("pos", r64 > 0))}
    avg = {k: A.total(R[m]) / A.const(cnt[k]) if cnt[k] else nan
           for k, m in (("neg", r64 < 0), ("nz", r64 != 0), ("pos", r64 > 0))}
    m2 = M2x / n
    constant = bool(np.all(x64 == x64[0]))
    thr = (EPS * float(mx)) ** 2
    flat = constant or float(m2) <= thr / FLAT_MARGIN
    free = not flat and float(m2) <= thr * FLAT_MARGIN
    skew = nan if flat or free else (S3 / n) / (m2 * A.sqrt(m2))
    kurt = nan if flat or free else (S4 / n) / (m2 * m2)
    vals = [total - one, cagr, _div(mx * sq252, sd_x), _div(mx * sq252, down), mdd, _div(cagr, abs(mdd)),
            avg["neg"], avg["nz"], avg["pos"], float(np.max(r64)), float(np.min(r64)), sd_r * sq252,
            mr - A.const(Z95) * sd_r, skew, kurt, _div(mx, sd_x)]
    out = np.empty(16, dtype=object if A is EXACT else LD)
    for k, v in enumerate(vals):
        out[k] = v
    if A is not LONGDOUBLE:
        return EvalRef(out)

    # ---- the bound (float64 arithmetic on the reference's own quantities)
    f = lambda v: float(v)
    Tc = (T + C_EV) * U
    w = (2 * T + C_EV) * U
    e_r, e_x = Tc * float(np.sum(np.abs(r64))) / T, Tc * float(np.sum(np.abs(x64))) / T
    B = np.zeros(16)
    lo = np.zeros(16)

    E2r, E2x = Tc * f(M2r) + 2 * T * e_r ** 2, Tc * f(M2x) + 2 * T * e_x ** 2

    def e_sd(M2, E2):
        s = np.sqrt(M2 / (T - 1))
        d = np.sqrt(E2 / (T - 1)) if M2 == 0 else min(np.sqrt(E2 / (T - 1)), E2 / (2 * np.sqrt(M2 * (T - 1))))
        return d + 2 * U * (s + d)

    Esd_r, Esd_x = e_sd(f(M2r), E2r), e_sd(f(M2x), E2x)
    # wealth
    E_cum = w * abs(f(total)) + 2 * U * abs(f(total - one))
    E_cagr = abs(f(total)) ** e * (e * w * 1.01 + 3 * U) + 2 * U * abs(f(cagr))
    nondecreasing = bool(np.all(r64 >= 0))
    E_dd = 0.0 if nondecreasing else 2 * w + 2 * U + U * abs(f(mdd))
    B[K["Cum. Return"]], B[K["CAGR"]], B[K["Max. DD"]] = E_cum, E_cagr, E_dd
    if f(mdd) == 0:
        B[K["Calmar"]] = 0.0
    elif E_dd < abs(f(mdd)) / 2:
        cal = abs(f(out[K["Calmar"]]))
        B[K["Calmar"]] = (E_cagr + cal * E_dd) / (abs(f(mdd)) - E_dd) + 2 * U * cal
    else:
        B[K["Calmar"]] = np.inf
    # Sharpe / per-period Sharpe
    s, mu = f(sd_x), f(mx)
    for name, scale in (("Sharpe", np.sqrt(252.0)), ("sharpe_per_period", 1.0)):
        k = K[name]
        if s == 0:
            B[k] = 0.0
            if mu != 0:
                B[k], lo[k] = np.inf, max(abs(mu) - e_x, 0.0) / Esd_x * scale * (1 - 4 * U)
        elif Esd_x < s / 2:
            B[k] = scale * (abs(mu) * Esd_x + s * e_x) / (s * (s - Esd_x)) + 3 * U * abs(f(out[k]))
        else:
            B[k] = np.inf
    D = f(down)
    if D > 0:
        dlt = Tc / 2 + 2 * U
        B[K["Sortino"]] = np.sqrt(252.0) * (e_x + abs(mu) * dlt / (1 - dlt)) / D + 3 * U * abs(f(out[K["Sortino"]]))
    for name, key in (("Avg. Loss", "neg"), ("Avg. Return", "nz"), ("Avg. Win", "pos")):
        if cnt[key]:
            m = {"neg": r64 < 0, "nz": r64 != 0, "pos": r64 > 0}[key]
            B[K[name]] = (cnt[key] + C_EV) * U * float(np.sum(np.abs(r64[m]))) / cnt[key]
    B[K["Ann. Vol."]] = np.sqrt(252.0) * Esd_r + 2 * U * abs(f(out[K["Ann. Vol."]]))
    B[K["Daily VaR"]] = e_r + Z95 * Esd_r + 2 * U * abs(f(out[K["Daily VaR"]]))
    if free:
        B[K["skew"]] = B[K["kurtosis"]] = np.inf
    elif not flat:
        M2 = f(M2x)
        rho = E2x / M2
        if rho > 0.1:
            B[K["skew"]] = B[K["kurtosis"]] = np.inf
        else:
            ab = np.abs(np.asarray(b, dtype=np.float64)) + e_x
            E3 = 3 * e_x * M2 + T * e_x ** 3 + Tc * float(np.sum(ab ** 3))
            E4 = 4 * e_x * abs(f(S3)) + 6 * e_x ** 2 * M2 + T * e_x ** 4 + Tc * float(np.sum(ab ** 4))
            m2f = M2 / T
            B[K["skew"]] = E3 / T / m2f ** 1.5 * (1 + 2 * rho) + abs(f(skew)) * (2 * rho + 6 * U)
            B[K["kurtosis"]] = E4 / T / m2f ** 2 * (1 + 3 * rho) + f(kurt) * (3 * rho + 6 * U)
    return EvalRef(out, B, lo)


# ------------------------------------------------------------------------------------------------- checking
def ratios(got, ref: EvalRef) -> np.ndarray:
    """|got - ref| / bound per statistic; < 1 passes.  inf where an exact output, a NaN or a +-inf differs (or a finite
    value where ``lo`` allows one is too small or has the wrong sign), 0 where there is no claim."""
    got = np.asarray(got, dtype=np.float64)
    out = np.zeros(16)
    for k in range(16):
        g, v, bnd = got[k], ref.values[k], ref.bound[k]
        v64 = float(v)
        if bnd == np.inf and not ref.lo[k] > 0:
            continue
        if np.isnan(v64) or np.isnan(g):
            out[k] = 0.0 if np.isnan(v64) and np.isnan(g) else np.inf
        elif np.isinf(v64):
            same = g == v64 or (ref.lo[k] > 0 and np.sign(g) == np.sign(v64) and abs(g) >= ref.lo[k])
            out[k] = 0.0 if same else np.inf
        elif np.isinf(g):
            out[k] = np.inf
        elif bnd == 0:
            out[k] = 0.0 if g == v64 else np.inf
        else:
            out[k] = float(abs(LD(g) - LD(v))) / bnd
    return out


# ------------------------------------------------------------------------------------------------- float64 emulation
def kernel_f64(r, x, years, fault=None, order="kernel", seed=0):
    """The kernel's float64 arithmetic on one series.  ``order`` = "kernel" (block_sum's order and 256 chunks),
    "forward" (sequential sums, one chunk) or "random" (a fresh permutation for every sum and a random chunk count).
    ``fault``: one of FAULTS, a seeded error for the tests that show the bound catches it."""
    assert fault is None or fault in FAULTS, fault
    r, x = np.asarray(r, dtype=np.float64), np.asarray(x, dtype=np.float64)
    T = len(r)
    n = float(T)
    rng = np.random.default_rng(seed)
    threads = {"kernel": THREADS, "forward": 1, "random": int(rng.integers(1, 1025))}[order]

    def total(v):
        v = np.asarray(v, dtype=np.float64)
        if order == "kernel":
            return kernel_sum(v) if len(v) else 0.0
        if order == "random":
            v = v[rng.permutation(len(v))]
        return float(np.cumsum(v)[-1]) if len(v) else 0.0

    neg, pos, nz = r < 0, r > 0, r != 0
    sr, sx = total(r), total(x)
    sneg, spos, snz = total(np.where(neg, r, 0.0)), total(np.where(pos, r, 0.0)), total(np.where(nz, r, 0.0))
    cneg, cpos, cnz = float(neg.sum()), float(pos.sum()), float(nz.sum())
    dn2 = total(np.where(x < 0, x * x, 0.0))
    lanes = np.arange(T) % THREADS
    seen = lanes < 128 if fault == "max_four_warps" else np.ones(T, dtype=bool)
    mx, mn = float(np.max(r[seen])), float(np.min(r[seen]))
    mr, mxs = sr / n, sx / n
    a, b = r - mr, x - mxs
    r2, x1, x2 = total(a * a), total(b), total(b * b)
    x3, x4 = total(b * b * b), total((b * b) * (b * b))

    # chunked scan of the wealth curve
    chunk = T // threads if fault == "chunk_floor" else -(-T // threads)
    i0 = np.minimum(np.arange(threads) * chunk, T)
    i1 = np.minimum(i0 + chunk, T)
    with np.errstate(invalid="ignore", over="ignore"):
        prod, lmax = np.ones(threads), np.full(threads, -np.inf)
        for j in range(chunk):
            live = i0 + j < i1
            idx = (i0 + j)[live]
            prod[live] = prod[live] * (1.0 + r[idx])
            lmax[live] = np.fmax(lmax[live], prod[live])
        cbase, cpeak = np.empty(threads), np.empty(threads)
        base, peak = 1.0, (1.0 if fault == "peak_starts_at_one" else -np.inf)
        for t in range(threads):
            cbase[t], cpeak[t] = base, peak
            peak = np.fmax(peak, base if fault == "peak_from_base" else base * lmax[t])
            base = base * prod[t]
        cum = cbase.copy()
        pk = np.full(threads, -np.inf) if fault == "chunk_peak_restart" else cpeak.copy()
        dd = np.full(threads, np.inf)
        for j in range(chunk):
            live = i0 + j < i1
            idx = (i0 + j)[live]
            cum[live] = cum[live] * (1.0 + r[idx])
            pk[live] = np.fmax(pk[live], cum[live])
            dd[live] = np.fmin(dd[live], cum[live] / pk[live])
    warps = (np.arange(threads) % THREADS) < 128 if fault == "max_four_warps" else np.ones(threads, dtype=bool)
    mdd = float(np.min(dd[warps])) - 1.0

    F = np.float64                        # IEEE division by zero, as on the device
    sr, mr, mxs, sneg, spos, snz, cneg, cpos, cnz, dn2, r2, x1, x2, x3, x4, base, mdd, n = map(
        F, (sr, mr, mxs, sneg, spos, snz, cneg, cpos, cnz, dn2, r2, x1, x2, x3, x4, base, mdd, n))
    with np.errstate(all="ignore"):
        ddof = n if fault == "ddof0" else n - 1.0
        sd_r, sd_x = np.sqrt(r2 / ddof), np.sqrt(x2 / ddof)
        cagr = np.power(abs(base), 1.0 / years) - 1.0
        down = np.sqrt(dn2 / (cneg if fault == "sortino_neg_count" else n))
        m2 = x2 / n
        m2c = (x2 - x1 * x1 / n) / n
        flat = fault != "no_flat_rule" and m2c <= (EPS * mxs) ** 2
        nan = float("nan")
        avg_ret = (sr / n) if fault == "avg_return_zeros" else (snz / cnz if cnz > 0 else nan)
        out = [base - 1.0, cagr, mxs / sd_x * np.sqrt(252.0), mxs / down * np.sqrt(252.0), mdd, cagr / abs(mdd),
               sneg / cneg if cneg > 0 else nan, avg_ret, spos / cpos if cpos > 0 else nan, mx, mn,
               sd_r * np.sqrt(252.0), sd_r * -Z95 + mr,
               nan if flat else (x3 / n) / (m2 * np.sqrt(m2)), nan if flat else (x4 / n) / (m2 * m2), mxs / sd_x]
    return np.array(out, dtype=np.float64)


# ------------------------------------------------------------------------------------------------- synthetic cases
# Each case is a list of calls (r [P][T], x [P][T], years).  Neighbouring series differ strongly in drift and spread,
# so a chunk that reads past its own series changes that series' wealth curve by about a percent.
def rf_daily(T):
    """A risk-free rate that moves every day (1-3 % a year), de-annualised as compute_excess_returns does."""
    rf = 0.02 + 0.01 * np.sin(np.arange(T) / 200.0)
    return (rf + 1.0) ** (1.0 / 252.0) - 1.0


def series(P, T, seed):
    rng = np.random.default_rng(seed)
    p = np.arange(P)
    scale = 0.004 * (1 + 3 * (p % 4))
    drift = 3e-4 * np.where(p % 2, -1.0, 2.0)
    r = drift[:, None] + scale[:, None] * rng.standard_normal((P, T))
    return r, r - rf_daily(T)


def years_of(T):
    return T / 252.0


def _chunk(T):
    return -(-T // THREADS)


def drawdown_at(T, peak, trough, seed, drop=0.3):
    """A rising curve (small noisy gains) whose running peak is the point after return ``peak`` and whose deepest
    point is after return ``trough``: a 5 % jump at ``peak``, a fall of ``drop`` spread over (peak, trough], gains after."""
    rng = np.random.default_rng(seed)
    r = 6e-4 + 1e-4 * rng.standard_normal(T)
    r[peak] = 0.05
    r[peak + 1:trough + 1] = (1.0 - drop) ** (1.0 / (trough - peak)) - 1.0
    return r


def _stack(rows, T):
    r = np.stack(rows)
    return r, r - rf_daily(T)


def lengths_case(T):
    return lambda: [series(4, T, 1000 + T) + ((2.0 / 365.0) if T == 2 else years_of(T),)]


def dd_across_chunks(T):
    """Peak = last return of chunk t, trough = first return of chunk t + 1, for chunks in the first and the second
    half of the threads and the last pair of non-empty chunks."""
    c = _chunk(T)
    last = (T - 1) // c
    ts = sorted({0, 31, 127, 128, 200, last - 1} & set(range(last)))
    rows = [drawdown_at(T, (t + 1) * c - 1, (t + 1) * c, 2000 + t) for t in ts]
    return lambda: [_stack(rows, T) + (years_of(T),)]


def dd_inside_chunk(T):
    c = _chunk(T)
    rows = [drawdown_at(T, t * c + 1, t * c + c - 2, 3000 + t) for t in (0, 100, 130, (T - 1) // c - 1)]
    return lambda: [_stack(rows, T) + (years_of(T),)]


def dd_shapes(T):
    """Peak at index 0 and trough at T - 1; a curve that declines from the first day (its peak is W_0, not 1); a
    global peak in the last return, and a trough there; a curve that never falls (zeros included)."""
    rng = np.random.default_rng(4000 + T)
    first_last = -4e-4 - np.abs(1e-4 * rng.standard_normal(T))
    first_last[0] = 0.05
    decline = -4e-4 - np.abs(1e-4 * rng.standard_normal(T))
    decline[0] = -0.02
    peak_last = drawdown_at(T, T - 3, T - 2, 4001)
    peak_last[T - 1] = 0.2
    trough_last = 6e-4 + 1e-4 * rng.standard_normal(T)
    trough_last[T - 1] = -0.4
    never = np.abs(1e-3 * rng.standard_normal(T))
    never[::5] = 0.0
    return lambda: [_stack([first_last, decline, peak_last, trough_last, never], T) + (years_of(T),)]


def wipe_out(T):
    """A -100 % day in the middle (and one in the last non-empty chunk) between ordinary days."""
    def make():
        r, _ = series(3, T, 5000 + T)
        r[0, T // 2] = -1.0
        r[1, T - 1] = -1.0
        return [(r, r - rf_daily(T), years_of(T))]
    return make


def insolvent(T, day):
    """Series that fall below -100 % on ``day`` and are passed through adjust_returns: with the wealth below 1 the
    adjusted day makes it negative (the tail is constant and negative), with the wealth above 1 tiny and positive."""
    def make():
        import pandas as pd
        from incorporating_different_sources_b200.evaluation import adjust_returns
        rng = np.random.default_rng(6000 + T)
        rows = []
        for drift in (-3e-3 * 60 / day, 4e-3 * 60 / day):
            v = drift + 2e-3 * rng.standard_normal(T)
            v[day] = -1.4
            rows.append(v)
        raw = np.stack(rows)
        rf = rf_daily(T)
        r = np.stack([adjust_returns(pd.Series(v)).to_numpy() for v in raw])
        x = np.stack([adjust_returns(pd.Series(v - rf)).to_numpy() for v in raw])
        return [(r, x, years_of(T))]
    return make


def conditional(T):
    """No losing day; no winning day; all zeros (returns and excess); zeros mixed in; no negative excess."""
    def make():
        rng = np.random.default_rng(7000 + T)
        g = 5e-3 * rng.standard_normal((5, T))
        r = np.stack([np.abs(g[0]) + 1e-4, -np.abs(g[1]) - 1e-4, np.zeros(T), g[3], g[4] + 1e-3])
        r[3, ::5] = 0.0
        r[3, 3::7] = 0.0
        x = r - rf_daily(T)
        x[2] = 0.0
        x[4] = np.abs(x[4])
        return [(r, x, years_of(T))]
    return make


def moments(T):
    """Near-symmetric excess returns (exact skew 0), one large outlier (kurtosis ~ T), a mean 10**3 and 10**6 times the
    spread, one value one ulp off a constant (below the flat threshold by far)."""
    def make():
        rng = np.random.default_rng(8000 + T)
        h = 1e-2 * rng.standard_normal(T // 2)
        sym = np.concatenate([h, -h, np.zeros(T % 2)])[rng.permutation(T)]
        out = 1e-3 * rng.standard_normal(T)
        out[T // 3] = 1.0
        big3 = 0.01 + 1e-5 * rng.standard_normal(T)
        big6 = 0.01 + 1e-8 * rng.standard_normal(T)
        ulp = np.full(T, 0.1)
        ulp[T // 2] = np.nextafter(0.1, 1.0)
        x = np.stack([sym, out, big3, big6, ulp])
        r = x + rf_daily(T)
        return [(r, x, years_of(T))]
    return make


# the flat series: the kernel's block-sum mean of the first four is off by 1 to 3 ulp (excess 0.1 x 4149, 3e-4 x 257
# and x 601, the de-annualised 2 % of a zero-return series x 4149); the others' block-sum mean is exact.
CONSTANTS = ((4149, 0.1), (257, 3e-4), (601, 3e-4), (4149, -((1.02 ** (1 / 252)) - 1)),
             (4149, 0.125), (256, 3e-4), (2, 0.1), (65536, 2.0 ** -10))


def constant_case(T, v):
    def make():
        rng = np.random.default_rng(9000 + T)
        x = np.full((1, T), v)
        r = np.zeros((1, T)) if v < 0 else 5e-3 * rng.standard_normal((1, T))
        return [(r, x, years_of(T))]
    return make


def ensemble(P, T):
    return lambda: [series(P, T, 10000 + P) + (years_of(T),)]


def years_case():
    r, x = series(4, 600, 11000)
    return [(r, x, y) for y in (2.0 / 365.0, 0.5, 2.38, 10.0, 40.0)]


LENGTHS = (2, 255, 256, 257, 511, 512, 513, 4149, 65536, 65537, 100003)
CASES = {f"length_{T}": lengths_case(T) for T in LENGTHS}
CASES.update({f"dd_across_chunks_{T}": dd_across_chunks(T) for T in (256, 513, 4149, 65537)})
CASES.update({f"dd_inside_chunk_{T}": dd_inside_chunk(T) for T in (4149, 65537)})
CASES.update({f"dd_shapes_{T}": dd_shapes(T) for T in (257, 512, 4149)})
CASES.update({f"wipe_out_{T}": wipe_out(T) for T in (257, 4149)})
CASES.update({"insolvent_257": insolvent(257, 200), "insolvent_4149": insolvent(4149, 3000)})
CASES.update({f"conditional_{T}": conditional(T) for T in (40, 513, 4149)})
CASES.update({f"moments_{T}": moments(T) for T in (257, 4149, 65536)})
CASES.update({f"constant_{T}_{v:.3g}": constant_case(T, v) for T, v in CONSTANTS})
CASES.update({"ensemble_1": ensemble(1, 4149), "ensemble_64": ensemble(64, 4149), "ensemble_3000": ensemble(3000, 513)})
CASES["years"] = years_case
