"""Extended-precision restatement and a-priori bound for the backtest loop body (loop_kernels.cu).

What the loop body computes (portfolio_calculations.py:1054-1075 turnover, :1077-1104 distance to the value-weighted
portfolio, :1127-1219 return, drift, renormalisation, cost and metrics; backtest.compute_portfolio_turnover):

  * Metrics of rebalance s over its members (``member[s]``, all columns without a mask), from W[s]:
    max_long / max_short = max / min of the positive / negative weights (NaN for an empty selection, as pandas' max),
    avg_long / avg_short = their means, distance = mean over the members of |scale w_i - cap_i / sum(caps)| with the
    caps of the rebalance row.
  * Segment s (1 <= s <= R; s = R is the tail up to ``last_row``): the days reb_row[s-1] + 1 .. reb_row[s], starting
    from W[s-1] on the HELD set ``member[s-1]``.  Columns outside the held set are never read.  On day d, with
    r_i = p_d,i / p_d-1,i - 1 (float64 on both sides) and rf_d = (1 + rf_row[d])^(1/252) - 1:
        r_d   = sum_i w_i r_i + (1 - sum_i w_i) rf_d          (skipna sums)
        w_i  <- w_i (1 + r_i) / (sum_i w_i (1 + r_i) + (1 - sum_i w_i)(1 + rf_d))
    A NaN return makes the weight NaN for the rest of the segment: it is skipped in the product sum at once, still
    counts in that day's sum_i w_i (its weight was not NaN yet) and is skipped in every sum after.
    On the rebalance day (not in the tail) the turnover against the new weights W[s] on member[s] is
        to = (sum_i |wb_i - wa_i| + |sum wb - sum wa|) / 2     (outer merge of both index sets, NaN / missing -> 0)
    and r_d -= bps / 10^4 to.
  * returns[d - reb_row[0] - 1] = r_d, turnover[s - 1] = to, metrics[s] = the five metrics.

:func:`restate` evaluates all of it with the arithmetic of a chosen number type: ``np.longdouble`` for the reference
(64-bit mantissa, 2**11 below the bound), float64 with a chosen summation order to show that the bound holds for any
order, and ``fractions.Fraction`` to show that the longdouble evaluation is itself accurate.  NaN is tracked as a mask
(``dead``), so the same code runs on Fractions.

The bound (u = 2**-53, a priori, not tuned to measured errors).  Any summation tree over n non-zero terms returns the
exact sum plus at most gamma_n = n u / (1 - n u) times the sum of the magnitudes; zeros add exactly.
  * Weights.  One day of drift rounds w_i (1 + r_i) twice and divides by a total formed from n held terms plus the
    risk-free term: a relative error of at most (n + c) u G, G = (sum |w_i||1 + r_i| + |1 - sum w|(1 + rf_d)) /
    |1 + r_p|.  The total is 1 + r_p (the book's own return), so it stays away from 0 and G is the book's leverage.
    Errors of earlier days add, so on day j of a segment (j = 1 on the day after the rebalance) the weights going in
    carry at most (j - 1)(n + c) u G of relative error.
  * Returns.  The day's own sums add (n + c) u M_d with
        M_d = sum_held |w_i| (|r_i| + |1 + r_i|) + |1 - sum w| (1 + rf_d),
    and the inherited weight error adds (j - 1)(n + c) u G sum |w_i r_i|, which is below (j - 1)(n + c) u M_d as long
    as the book moves less than its own value in a day (sum |w_i r_i| < |1 + r_p|, true by orders of magnitude in
    every case here).  Hence
        |E(r_d)| <= (j + 1)(n + c) u M_d.
    CUDA's pow is within 2 ulp, and every O(1) rounding outside the sums (1 + r_i, the products, 1 - sum w, the
    division, the subtractions) is charged to c.
  * Turnover: the same form with sum |wb| + sum |wa| as the magnitude (wb carries the drift error of the whole
    segment, wa none); the rebalance-day return adds bps / 10^4 times that bound.
  * avg_long / avg_short: (n + c) u times sum |w| / count.  The distance divides by a cap sum of n terms before it
    sums n terms: (2 n + c) u times sum (scale |w_i| + cap_i / sum caps) / n.
  * max_long / max_short involve no arithmetic: they must equal the reference bit for bit.
c = 16 (C_LOOP) covers the O(1) roundings (at most eight per day plus pow's two ulp), with room to spare.
"""
from __future__ import annotations

from dataclasses import dataclass
from fractions import Fraction
from typing import Optional

import numpy as np

U = 2.0 ** -53
LD = np.longdouble
C_LOOP = 16
METRICS = ("max_long", "max_short", "avg_long", "avg_short", "distance")
FAULTS = ("drift_from_rebalance_day", "held_is_new_member", "no_rf_leg", "rf_365", "no_rf_turnover",
          "cost_day_after", "nan_weight_counts", "capsum_all_columns", "max_warp0_only")


def require_extended_precision():
    if np.finfo(LD).nmant < 63:
        raise RuntimeError("np.longdouble is not 80-bit extended precision on this platform: the reference needs it")


@dataclass
class LoopInputs:
    """The arguments of ``bp_backtest_batched`` as NumPy arrays: the market rows the loop reads and the call's own."""
    prices: np.ndarray                  # [D][N]
    caps: np.ndarray                    # [D][N]
    rf_row: np.ndarray                  # [D]
    reb_row: np.ndarray                 # [R] ascending, >= 1
    W: np.ndarray                       # [R][N]
    member: Optional[np.ndarray]        # [R][N] or None (= every column)
    last_row: int
    scale: float = 1.0
    bps: float = 0.0

    @property
    def N(self):
        return self.W.shape[1]

    @property
    def R(self):
        return self.W.shape[0]

    def members(self, s):
        """Boolean [N] mask of rebalance s's universe."""
        if self.member is None:
            return np.ones(self.N, dtype=bool)
        return np.asarray(self.member[s]) != 0


@dataclass
class LoopRef:
    """Reference outputs (number type of the evaluation) and, for the longdouble run, their bounds (float64)."""
    returns: np.ndarray
    turnover: np.ndarray
    metrics: np.ndarray
    b_returns: Optional[np.ndarray] = None
    b_turnover: Optional[np.ndarray] = None
    b_metrics: Optional[np.ndarray] = None


# ------------------------------------------------------------------------------------------------- number types
class _LD:
    @staticmethod
    def cv(x):
        return np.asarray(x, dtype=np.float64).astype(LD)

    @staticmethod
    def rf_daily(rf):
        return (LD(1) + LD(rf)) ** (LD(1) / LD(252)) - LD(1)

    @staticmethod
    def rf_daily_365(rf):
        return (LD(1) + LD(rf)) ** (LD(1) / LD(365)) - LD(1)

    @staticmethod
    def total(x):
        return np.sum(np.asarray(x, dtype=LD), dtype=LD) if len(x) else LD(0)

    const = staticmethod(LD)


class _F64:
    """float64 arithmetic; ``order`` = "kernel" (per-thread strided partials, then the warp and block shuffle trees of
    block_sum), "forward", "reverse" or "random" (a fresh permutation for every sum)."""

    def __init__(self, order="kernel", seed=0):
        self.order = order
        self.rng = np.random.default_rng(seed)

    @staticmethod
    def cv(x):
        return np.asarray(x, dtype=np.float64)

    @staticmethod
    def rf_daily(rf):
        return float(np.power(1.0 + float(rf), 1.0 / 252.0)) - 1.0

    @staticmethod
    def rf_daily_365(rf):
        return float(np.power(1.0 + float(rf), 1.0 / 365.0)) - 1.0

    const = staticmethod(float)

    def total(self, x):
        x = np.asarray(x, dtype=np.float64)
        if len(x) == 0:
            return 0.0
        if self.order == "forward":
            return float(np.cumsum(x)[-1])
        if self.order == "reverse":
            return float(np.cumsum(x[::-1])[-1])
        if self.order == "random":
            return float(np.cumsum(x[self.rng.permutation(len(x))])[-1])
        return kernel_sum(x)


class _Frac:
    @staticmethod
    def cv(x):
        return np.array([Fraction(float(v)) for v in np.ravel(x)], dtype=object).reshape(np.shape(x))

    @staticmethod
    def rf_daily(rf):
        # the exact evaluation takes the longdouble reference's rf_d as its input: pow is not rational
        return Fraction(*_LD.rf_daily(rf).as_integer_ratio())

    @staticmethod
    def total(x):
        return sum(list(x), Fraction(0))

    const = staticmethod(Fraction)


LONGDOUBLE = _LD()
FRACTION = _Frac()


def kernel_sum(x: np.ndarray, threads: int = 256) -> float:
    """float64 sum of x (entry i held by thread i % 256, slot i // 256) in the order of loop_kernels.cu: each thread adds
    its slots in turn, warp_sum's xor tree (offsets 16 .. 1) runs in every warp, then warp 0 adds the warp sums with
    the same tree."""
    n = len(x)
    per = -(-n // threads)
    a = np.zeros(per * threads)
    a[:n] = x
    a = a.reshape(per, threads)
    v = a[0].copy()
    for e in range(1, per):
        v = v + a[e]

    def warp_tree(v):                       # v [k][32]
        lanes = np.arange(32)
        for o in (16, 8, 4, 2, 1):
            v = v + v[:, lanes ^ o]
        return v[:, 0]

    ws = warp_tree(v.reshape(threads // 32, 32))
    last = np.zeros((1, 32))
    last[0, :len(ws)] = ws
    return float(warp_tree(last)[0])


# ------------------------------------------------------------------------------------------------- restatement
def _metrics(inp: LoopInputs, s: int, A, fault):
    """Five metrics of rebalance s (values of A's type) and their bounds."""
    mem = inp.members(s)
    idx = np.nonzero(mem)[0]
    w64 = np.asarray(inp.W[s], dtype=np.float64)
    wm = w64[idx]
    pos, neg = wm > 0, wm < 0
    if fault == "max_warp0_only":
        lane0 = (idx % 256) < 32
        pos_mx, neg_mn = pos & lane0, neg & lane0
    else:
        pos_mx, neg_mn = pos, neg
    nan = float("nan")
    mx = float(np.max(wm[pos_mx])) if pos_mx.any() else nan
    mn = float(np.min(wm[neg_mn])) if neg_mn.any() else nan
    nl, ns = int(pos.sum()), int(neg.sum())
    w = A.cv(wm)
    al = A.total(w[pos]) / A.const(nl) if nl else nan
    as_ = A.total(w[neg]) / A.const(ns) if ns else nan
    cap_idx = np.arange(inp.N) if fault == "capsum_all_columns" else idx
    row = inp.caps[int(inp.reb_row[s])]
    capsum = A.total(A.cv(row[cap_idx]))
    vw = A.cv(row[idx]) / capsum
    scale = A.const(float(inp.scale))
    n = len(idx)
    dist = A.total(np.abs(w * scale - vw)) / A.const(n) if n else nan
    vals = [mx, mn, al, as_, dist]
    with np.errstate(invalid="ignore", divide="ignore"):
        vw64 = row[idx] / np.sum(row[idx]) if n else np.zeros(0)
        b = [0.0, 0.0,
             (nl + C_LOOP) * U * float(np.sum(np.abs(wm[pos]))) / nl if nl else 0.0,
             (ns + C_LOOP) * U * float(np.sum(np.abs(wm[neg]))) / ns if ns else 0.0,
             (2 * n + C_LOOP) * U * float(np.sum(abs(inp.scale) * np.abs(wm) + np.abs(vw64))) / n if n else 0.0]
    return vals, b


def restate(inp: LoopInputs, A=LONGDOUBLE, fault: Optional[str] = None) -> LoopRef:
    """The loop body on ``inp`` in the arithmetic of ``A`` (LONGDOUBLE, FRACTION or an ``_F64``), optionally with one
    seeded fault (FAULTS) for the tests that show the bound catches it."""
    assert fault is None or fault in FAULTS, fault
    R, N = inp.R, inp.N
    reb = np.asarray(inp.reb_row, dtype=np.int64)
    T = int(inp.last_row - reb[0])
    dt = object if A is FRACTION else (LD if A is LONGDOUBLE else np.float64)
    rets = np.empty(T, dtype=dt)
    turn = np.empty(max(R - 1, 0), dtype=dt)
    met = np.empty((R, 5), dtype=dt)
    b_rets, b_turn, b_met = np.zeros(T), np.zeros(max(R - 1, 0)), np.zeros((R, 5))
    for s in range(R):
        vals, b = _metrics(inp, s, A, fault)
        for k in range(5):
            met[s, k] = vals[k]
        b_met[s] = b
    one, bps = A.const(1.0), A.const(float(inp.bps)) / A.const(10000.0)
    rf_fn = A.rf_daily_365 if fault == "rf_365" else A.rf_daily
    P = np.asarray(inp.prices, dtype=np.float64)
    late_cost = []                                        # fault "cost_day_after": (day index, cost)
    for s in range(1, R + 1):
        tail = s == R
        h = np.nonzero(inp.members(s if fault == "held_is_new_member" and not tail else s - 1))[0]
        n = len(h)
        w = A.cv(np.asarray(inp.W[s - 1], dtype=np.float64)[h])
        dead = np.zeros(n, dtype=bool)                    # NaN weight (a NaN return earlier in the segment)
        end = int(inp.last_row if tail else reb[s])
        first = int(reb[s - 1]) + (0 if fault == "drift_from_rebalance_day" else 1)
        for d in range(first, end + 1):
            with np.errstate(invalid="ignore", divide="ignore"):
                r64 = P[d, h] / P[d - 1, h] - 1.0         # pct_change, float64 on both sides
            nan_today = np.isnan(r64) & ~dead
            if fault == "nan_weight_counts":
                r64 = np.where(np.isnan(r64), 0.0, r64)
                nan_today[:] = False
            live = ~dead & ~nan_today
            r64 = np.where(live, r64, 0.0)
            r = A.cv(r64)
            pr = A.total((w * r)[live])
            sw = A.total(w[~dead])
            rf_d = rf_fn(inp.rf_row[d])
            rd = pr if fault == "no_rf_leg" else pr + (one - sw) * rf_d
            # magnitude of the day (weights going in), for the bound
            w_in = np.where(dead, 0.0, np.abs(np.asarray(w, dtype=np.float64)))
            M = float(np.sum(w_in * (np.abs(r64) + np.abs(1.0 + r64)))) \
                + abs(1.0 - float(sw)) * (1.0 + abs(float(rf_d)))
            upd = (one - sw) * (one + rf_d)
            w = np.where(live, w * (one + r), w)
            dead = dead | nan_today
            w = w / (A.total(w[~dead]) + upd)
            if d <= reb[s - 1]:
                continue                                  # the faulty extra drift on the rebalance day itself
            j = d - int(reb[s - 1])
            b = (j + 1) * (n + C_LOOP) * U * M
            k = d - int(reb[0]) - 1
            if d == end and not tail:
                new = inp.members(s)
                wa64 = np.where(new, np.asarray(inp.W[s], dtype=np.float64), 0.0)
                wa64 = np.where(np.isnan(wa64), 0.0, wa64)
                held_full = np.zeros(N, dtype=bool)
                held_full[h] = True
                union = np.nonzero(new | held_full)[0]
                wb = A.cv(np.zeros(N))
                wb[h[~dead]] = w[~dead]
                wa = A.cv(wa64)
                diff = A.total(np.abs(wb[union] - wa[union]))
                sb, sa = A.total(wb[union]), A.total(wa[union])
                to = diff / A.const(2.0) if fault == "no_rf_turnover" else (diff + abs(sb - sa)) / A.const(2.0)
                turn[s - 1] = to
                mag = float(np.sum(np.abs(np.asarray(w, dtype=np.float64)[~dead]))) + float(np.sum(np.abs(wa64)))
                b_turn[s - 1] = (j + 1) * (len(union) + C_LOOP) * U * mag
                b += float(inp.bps) / 1e4 * b_turn[s - 1] + 2 * U * float(inp.bps) / 1e4 * abs(float(to))
                if fault == "cost_day_after":
                    late_cost.append((k + 1, bps * to))
                else:
                    rd = rd - bps * to
            rets[k] = rd
            b_rets[k] = b
    for k, c in late_cost:
        if k < T:
            rets[k] = rets[k] - c
    return LoopRef(rets, turn, met, b_rets, b_turn, b_met)


# ------------------------------------------------------------------------------------------------- checking
def ratio(got, ref_vals, bound) -> float:
    """max |got - ref| / bound over the entries; NaN must sit exactly where the reference has NaN, and an entry whose
    bound is 0 must match exactly.  < 1 passes."""
    got = np.asarray(got, dtype=np.float64)
    ref64 = np.asarray(ref_vals, dtype=np.float64)
    bound = np.asarray(bound, dtype=np.float64)
    assert got.shape == ref64.shape, (got.shape, ref64.shape)
    if not np.array_equal(np.isnan(got), np.isnan(ref64)):
        return np.inf
    m = ~np.isnan(ref64)
    if not m.any():
        return 0.0
    err = np.abs(got[m].astype(LD) - np.asarray(ref_vals)[m].astype(LD)).astype(np.float64)
    bnd = bound[m]
    if not np.all(np.isfinite(err)) or np.any((bnd == 0) & (err != 0)):
        return np.inf
    with np.errstate(invalid="ignore", divide="ignore"):
        return float(np.max(np.where(bnd > 0, err / bnd, 0.0)))


def ratios(got, ref: LoopRef) -> dict:
    """Worst |E| / bound of each output of a run (returns, turnover, metrics); max_long / max_short must be bit-exact
    (ratio inf otherwise, 0 when equal)."""
    rets, turn, met = (np.asarray(x, dtype=np.float64) for x in got)
    out = {"returns": ratio(rets, ref.returns, ref.b_returns), "turnover": ratio(turn, ref.turnover, ref.b_turnover)}
    ref_met = np.asarray(ref.metrics, dtype=np.float64)
    for k, name in enumerate(METRICS):
        if k < 2:
            exact = np.array_equal(met[:, k], ref_met[:, k], equal_nan=True)
            out[name] = 0.0 if exact else np.inf
        else:
            out[name] = ratio(met[:, k], ref.metrics[:, k], ref.b_metrics[:, k])
    return out


# ------------------------------------------------------------------------------------------------- synthetic cases
def market(D: int, N: int, seed: int):
    """Seeded daily prices (1-3 % daily moves), caps and a risk-free row that changes every day (0.5-6 % a year)."""
    rng = np.random.default_rng(seed)
    vol = rng.uniform(0.01, 0.03, N)
    P = rng.uniform(20.0, 400.0, N) * np.cumprod(1.0 + vol * rng.standard_normal((D, N)), axis=0)
    caps = P * rng.uniform(5e7, 5e9, N)
    rf = 0.005 + 0.055 * rng.random(D)
    return P, caps, rf


def changing_members(R: int, N: int, seed: int, frac: float = 0.7) -> np.ndarray:
    """[R][N] masks that change at most rebalances: about a tenth of the columns leave or enter at each one, and about
    a fifth of the columns are never members."""
    rng = np.random.default_rng(seed)
    never = rng.random(N) < 0.2
    if never.all():
        never[0] = False
    m = (rng.random(N) < frac) & ~never
    out = np.zeros((R, N), dtype=np.uint8)
    for s in range(R):
        if s and rng.random() < 0.85:
            flip = (rng.random(N) < 0.1) & ~never
            m = m ^ flip
        if not m.any():
            m[np.nonzero(~never)[0][0]] = True
        out[s] = m
    return out


SUMS = (0.3, 1.0, 2.5)


def weights(member: Optional[np.ndarray], R: int, N: int, seed: int) -> np.ndarray:
    """[R][N] weights that make every term of the loop visible: long/short books with sum w at 0.3, 1 and 2.5, every
    fourth rebalance all long or all short, about a tenth of the member weights exactly 0, and the largest and the most
    negative weight in the first member columns, in columns >= 32 or in columns >= 256, by turn.  Non-members get 0."""
    rng = np.random.default_rng(seed)
    W = np.zeros((R, N))
    for s in range(R):
        cols = np.arange(N) if member is None else np.nonzero(member[s])[0]
        n = len(cols)
        if n == 0:
            continue
        kind = ("ls", "ls", "ls", "long" if s % 8 == 3 else "short")[s % 4]
        target = SUMS[s % 3]
        raw = rng.standard_normal(n) * (2.0 / n)
        if kind == "long":
            w = np.abs(raw) + 1e-3 / n
            w *= target / w.sum()
        elif kind == "short":
            w = -np.abs(raw) - 1e-3 / n
            w *= target / -w.sum()
        else:
            w = raw + (target - raw.sum()) / n
        if n == 1:
            W[s, cols] = w if s % 4 != 2 else -w
            continue
        w[rng.random(n) < 0.1] = 0.0
        # where the extremes sit: first member columns, columns >= 32, columns >= 256 (when there are such members)
        where = s % 3
        lo = {0: 0, 1: 32, 2: 256}[where]
        cand = np.nonzero(cols >= lo)[0]
        if len(cand) < 2:
            cand = np.arange(n)
        big = 1.5 * np.max(np.abs(w)) + 1.0 / n
        if kind in ("ls", "long"):
            w[cand[0]] = big
        if kind in ("ls", "short"):
            w[cand[0] if kind == "short" else cand[1] if where == 0 else cand[-1]] = -big
        W[s, cols] = w
    return W


def case(N: int, D: int, reb_row, last_row: int, seed: int, member="changing", scale: float = 5.0,
         bps: float = 15.0, holes=()) -> LoopInputs:
    """A full loop input.  ``member``: "changing", None (no mask) or "one" (one stock at each rebalance, moving).
    ``holes``: (segment s, day offset k, days) = NaN prices in the highest held column with a non-zero weight of
    segment s from row reb_row[s-1] + k on, for ``days`` rows (a halt) or, with days None, to the end of the data (a
    delisting: the column leaves every later universe)."""
    P, caps, rf = market(D, N, seed)
    reb = np.asarray(reb_row, dtype=np.int32)
    R = len(reb)
    if isinstance(member, str) and member == "changing":
        mem = changing_members(R, N, seed + 1)
    elif isinstance(member, str) and member == "one":
        mem = np.zeros((R, N), dtype=np.uint8)
        mem[np.arange(R), np.arange(R) % N] = 1
    else:
        mem = member
    W = weights(mem, R, N, seed + 2)
    for seg, k, days in holes:
        held = np.ones(N, dtype=bool) if mem is None else mem[seg - 1] != 0
        c = int(np.nonzero(held & (W[seg - 1] != 0))[0][-1])
        a = int(reb[seg - 1]) + k
        if days is None:
            P[a:, c] = np.nan
            mem[seg:, c] = 0
            W[seg:, c] = 0.0
        else:
            P[a:a + days, c] = np.nan
    return LoopInputs(P, caps, rf, reb, W, mem, int(last_row), scale, bps)


def held_rows(inp: LoopInputs):
    """Per column, the price rows and the caps rows the loop may read: the rows of the segments in which it is held
    (the rebalance row before the segment included) and the rebalance rows at which it is a member."""
    D, N = inp.prices.shape
    pr = np.zeros((D, N), dtype=bool)
    cr = np.zeros((D, N), dtype=bool)
    reb = np.asarray(inp.reb_row)
    for s in range(inp.R):
        cr[reb[s]] |= inp.members(s)
        end = inp.last_row if s == inp.R - 1 else reb[s + 1]
        pr[reb[s]:end + 1] |= inp.members(s)[None, :]
    return pr, cr


def poisoned(inp: LoopInputs) -> LoopInputs:
    """The same call with every value the loop must not read replaced: NaN and +-inf prices and caps of 1e300 outside
    the rows of ``held_rows``, NaN weights outside each rebalance's members."""
    pr, cr = held_rows(inp)
    bad = np.resize(np.array([np.nan, np.inf, -np.inf]), inp.prices.size).reshape(inp.prices.shape)
    mem = np.stack([inp.members(s) for s in range(inp.R)])
    return LoopInputs(np.where(pr, inp.prices, bad), np.where(cr, inp.caps, 1e300), inp.rf_row, inp.reb_row,
                      np.where(mem, inp.W, np.nan), inp.member, inp.last_row, inp.scale, inp.bps)


# ------------------------------------------------------------------------------------------------- the cases
# Widths at the edges of the kernel's lanes, warps and register slots (asset i sits in thread i % 256, slot i // 256;
# 2048 = 8 slots x 256 threads is the limit).
WIDTHS = (1, 31, 32, 33, 255, 256, 257, 500, 1024, 1792, 1793, 2047, 2048)
COSTS = (0.0, 15.0, 1000.0)
SCALES = (1.0, 5.0)


def width_case(N: int) -> LoopInputs:
    """Six rebalances (a 1-day segment, 5- to 22-day ones) and a 14-day tail on a mask that changes at most of them."""
    k = WIDTHS.index(N) if N in WIDTHS else N
    return case(N, 70, [3, 4, 9, 14, 30, 52], 66, seed=100 + N, scale=SCALES[k % 2], bps=COSTS[k % 3])


SEGMENT_CASES = {          # N = 300: slots 0 and 1 of every thread hold data
    "daily": lambda: case(300, 50, np.arange(1, 41), 45, seed=201, bps=15.0),
    "weekly": lambda: case(300, 125, np.arange(3, 120, 5), 122, seed=202, scale=1.0, bps=15.0),
    "monthly": lambda: case(300, 260, np.arange(2, 250, 21), 255, seed=203, bps=1000.0),
    "day_next_to_200_days": lambda: case(300, 220, [10, 11, 211], 215, seed=204, bps=15.0),
    "single_rebalance": lambda: case(300, 70, [20], 60, seed=205),
    "no_tail": lambda: case(300, 40, [5, 12, 30], 30, seed=206, bps=1000.0),
    "tail_120_days": lambda: case(300, 140, [3, 10], 130, seed=207, scale=1.0),
    "first_row_1": lambda: case(300, 30, [1, 6, 20], 25, seed=208, bps=15.0),
    "no_mask": lambda: case(257, 60, [2, 9, 10, 31], 50, seed=209, member=None, bps=15.0),
    "one_stock_universe": lambda: case(40, 60, [2, 9, 10, 31, 40], 50, seed=210, member="one", bps=1000.0),
}


def hole_case() -> LoopInputs:
    """Price holes in held columns: a one-day halt on the day after a rebalance (which is itself the next rebalance
    day), a two-day halt inside a segment, and a delisting in the middle of a 30-day segment."""
    return case(300, 120, [5, 6, 11, 30, 31, 60, 90], 115, seed=211, bps=1000.0,
                holes=[(1, 1, 1), (4, 7, 2), (6, 10, None)])


def oracle_inputs(spec, mkt, md, start, end) -> LoopInputs:
    """The loop's inputs of ``backtest_portfolio(spec, start, end, md)`` laid out as backtest._batched_weights lays them
    out, without the engine: universes from select_universes (host only), each date's weights from the oracle in the
    universe's cap order, 0 outside it.  ``mkt`` must hold the same prices as ``md`` (the oracle reads it)."""
    import pandas as pd
    from incorporating_different_sources_b200.backtest import get_window_trading_days, rebalance_flags, select_universes
    from incorporating_different_sources_b200.windows import HF_LOOKBACK_DAYS
    from oracle import bayes_oracle as bo
    prices_df = md["stock_prices_df"]
    dates = prices_df.index
    in_range = np.nonzero((dates >= pd.Timestamp(start)) & (dates <= pd.Timestamp(end)))[0]
    reb_pos = in_range[rebalance_flags(dates[in_range], spec["rebalancing_frequency"])]
    universes, _, _ = select_universes(md["stock_market_caps_df"], prices_df, md["stock_intraday_prices_df"],
                                       dates[reb_pos], spec["size"], get_window_trading_days(spec),
                                       spec["rebalancing_frequency"],
                                       lookback_days=HF_LOOKBACK_DAYS.get(spec["rolling_window_frequency"]))
    col_pos = {c: i for i, c in enumerate(prices_df.columns)}
    R, N = len(reb_pos), len(prices_df.columns)
    W = np.zeros((R, N))
    member = np.zeros((R, N), dtype=np.uint8)
    for r, names in enumerate(universes):
        cols = np.array([col_pos[n] for n in names])
        W[r, cols], _ = bo.window_weights(spec, mkt, int(reb_pos[r]), cols=cols)
        member[r, cols] = 1
    scale = spec["risk_aversion"] if spec.get("risk_aversion") is not None else 1
    return LoopInputs(prices_df.to_numpy(dtype=np.float64), mkt.caps, mkt.rf, reb_pos.astype(np.int32), W, member,
                      int(in_range[-1]), float(scale), float(spec["turnover_cost"]))
