"""Host-side integer work of the path: which rows make up each rebalance window.

Everything here is index arithmetic on dates and must be bit-exact with the reference
(SURVEY.md H6): ``rolling_window`` counts PRICES so a window has n-1 returns (F2,
``portfolio_calculations.py:159,:60``); the risk-free exponent uses the window's own calendar
span (F3, ``:40-41``); the intraday window is ``(d - D + 1 day, d + 1 day]`` with the first bar's
return dropped (F5, ``:310-314``).
"""
from __future__ import annotations

from dataclasses import dataclass
from typing import Optional, Sequence

import numpy as np

_DAY = np.timedelta64(1, "D")
HF_LOOKBACK_DAYS = {"daily": 1, "weekly": 7, "monthly": 31}     # portfolio_calculations.py:299-304


@dataclass
class WindowBatch:
    """One batch of rebalance windows sharing a ``portfolio_spec`` (mirrors ``bp_window_batch``)."""
    rolling_window: int
    day_row: np.ndarray          # int32 [W] row of the trade date in the uploaded daily arrays
    span_days: np.ndarray        # int32 [W] calendar days first -> last window date
    hf_lo: Optional[np.ndarray]  # int32 [W] intraday price rows [lo, hi)
    hf_hi: Optional[np.ndarray]
    mcm_index: int = 0
    mcm_scaling: float = 1.0
    risk_aversion: float = 1.0
    prior_weights: int = 0       # 0 value weighted, 1 equally weighted
    mcm_rows: int = 0            # MCM observations averaged (0 = rolling_window)
    prior_n: Optional[np.ndarray] = None   # injected conjugate_prior_n per window
    resampled: bool = False      # weekly windows: rows refer to the ResampledRows of plan_weekly_windows
    extra_row: Optional[np.ndarray] = None   # int32 [W] per-date last return row (weekly windows)
    caps_row: Optional[np.ndarray] = None    # int32 [W] daily row of the trade date (weekly windows)

    @property
    def n_windows(self) -> int:
        return int(self.day_row.shape[0])


def mcm_index_of(strategy: str) -> int:
    """Column of the uploaded MCM block: 0 = VIX, 1 = EPU (dispatcher at :1012-1028)."""
    if "vix" in strategy:
        return 0
    if "epu" in strategy:
        return 1
    return 0


def prior_kind_of(strategy: str) -> int:
    """``calculate_conjugate_prior_w`` (:369-378): 'vw' is tested before 'ew'."""
    if "vw" in strategy:
        return 0
    if "ew" in strategy:
        return 1
    raise ValueError("Unknown conjugate portfolio prior weights.")


def hf_lookback(spec, hf_lookback_days: Optional[int] = None) -> int:
    if hf_lookback_days is not None:
        return int(hf_lookback_days)
    freq = spec["rolling_window_frequency"]
    if freq not in HF_LOOKBACK_DAYS:
        raise RuntimeError("Unknown rolling window frequency.")               # :308
    return HF_LOOKBACK_DAYS[freq]


def plan_daily_windows(spec, dates: np.ndarray, d_indices: Sequence[int], hf_ts: Optional[np.ndarray] = None,
                       hf_lookback_days: Optional[int] = None, need_hf: bool = True,
                       row_offset: int = 0, hf_row_offset: int = 0) -> WindowBatch:
    """Window descriptors for ``rolling_window_frequency == 'daily'``.

    ``dates`` is the (sorted) business-day index of the uploaded daily arrays, ``d_indices`` the
    positions of the trade dates in it.  ``row_offset`` / ``hf_row_offset`` shift the produced row
    numbers when only a slice of the market (a rank's date shard plus halo) is resident.
    """
    n = int(spec["rolling_window"])
    d_idx = np.asarray(d_indices, dtype=np.int64)
    if d_idx.ndim != 1 or d_idx.size == 0:
        raise ValueError("need at least one trade date")
    if d_idx.min() < n - 1:
        raise ValueError(f"a window of {n} prices needs {n - 1} rows before the trade date")
    first = d_idx - (n - 1)
    days = dates.astype("datetime64[D]").astype(np.int64)
    span = days[d_idx] - days[first]
    # the reference asserts max gap <= mean gap + 4 inside every window (:40-44)
    gaps = np.diff(days)
    win_gaps = np.lib.stride_tricks.sliding_window_view(gaps, n - 1)[first]
    assert np.all(win_gaps.max(axis=1) <= span / (n - 1) + 4), "Unexpected large gap between return dates."
    hf_lo = hf_hi = None
    if need_hf:
        if hf_ts is None:
            raise ValueError("intraday timestamps required for the conjugate prior")
        D = hf_lookback(spec, hf_lookback_days)
        d = dates[d_idx]
        start = d - D * _DAY + _DAY                                              # :310-311
        hf_lo = np.searchsorted(hf_ts, start, side="right")
        hf_hi = np.searchsorted(hf_ts, d + _DAY, side="right")                   # :312
        hf_lo = (hf_lo - hf_row_offset).astype(np.int32)
        hf_hi = (hf_hi - hf_row_offset).astype(np.int32)
    strat = spec["weighting_strategy"]
    conj = strat.startswith("conjugate")
    return WindowBatch(
        rolling_window=n,
        day_row=(d_idx - row_offset).astype(np.int32),
        span_days=span.astype(np.int32),
        hf_lo=hf_lo, hf_hi=hf_hi,
        mcm_index=mcm_index_of(strat) if conj else 0,
        mcm_scaling=float(spec["mcm_scaling"]) if conj and spec.get("mcm_scaling") is not None else 1.0,
        risk_aversion=float(spec["risk_aversion"]) if spec.get("risk_aversion") is not None else 1.0,
        prior_weights=prior_kind_of(strat) if conj else 0,
    )


def plan_wave_fractions(hf_hi: np.ndarray, n_hf_rows: int, wave: int, max_segments: int = 8, tail_split: int = 1):
    """Cut points of a segmented intraday upload for a date-sorted conjugate batch (``bp_set_upload_fractions``):
    whole solver waves of windows per segment (several per segment when there are more waves than segments), then the
    remainder of the batch as ``tail_split`` segments.  Between segments the library solves full waves only (a solver
    launch costs the latency of one factorisation however few windows it has); before the LAST segment it solves
    everything that is ready.  Cutting the remainder in two or three so that less work follows the copy was measured on
    the C2 workload (tools/e2e_tail.py): 29.00 ms (one tail segment) / 29.55 (two) / 29.41 (three) -- the short launches
    are too inefficient, the GPU falls behind the bus -- hence the default of 1.  Returns the cumulative row fractions,
    or ``None`` when the batch is too small or not sorted by date."""
    hi = np.asarray(hf_hi, dtype=np.int64)
    W = int(hi.shape[0])
    if wave <= 0 or W < 2 * wave or max_segments < 2 or np.any(np.diff(hi) < 0):
        return None
    full = W // wave
    rest = W - full * wave
    n_tail = max(1, min(int(tail_split), max_segments - 1)) if rest >= 128 * max(1, int(tail_split)) else (1 if rest > 0 else 0)
    per = -(-full // max(1, max_segments - n_tail))
    counts = [per * wave] * (full // per)
    if full % per:
        counts.append((full % per) * wave)
    for k in range(n_tail):
        counts.append(rest // n_tail + (1 if k < rest % n_tail else 0))
    ends = np.cumsum(counts)
    return [float(hi[e - 1]) / float(n_hf_rows) for e in ends]


def slice_batch(batch: WindowBatch, i0: int, i1: int) -> WindowBatch:
    """Windows [i0, i1) of a batch (views of the per-window arrays, same scalars)."""
    import dataclasses
    cut = lambda a: None if a is None else a[i0:i1]
    return dataclasses.replace(batch, day_row=batch.day_row[i0:i1], span_days=batch.span_days[i0:i1], hf_lo=cut(batch.hf_lo),
                               hf_hi=cut(batch.hf_hi), prior_n=cut(batch.prior_n), extra_row=cut(batch.extra_row),
                               caps_row=cut(batch.caps_row))


def split_batch_by_fractions(batch: WindowBatch, cum_fractions: Sequence[float], n_hf_rows: int):
    """Cut a date-sorted conjugate batch along the segment boundaries of a segmented upload
    (``plan_wave_fractions``): sub-batch k holds the windows whose last intraday row lies in segment k.  Evaluated one
    after the other behind an asynchronous upload, sub-batch k only waits for segments <= k (``wait_hf_rows`` in the
    library), so its compute overlaps the copy of the later segments -- on every path, including the pre-summed day
    blocks of long look-backs, which are not pipelined inside one call.  Returns [(i0, i1, sub_batch), ...]."""
    hi = np.asarray(batch.hf_hi, dtype=np.int64)
    if np.any(np.diff(hi) < 0):
        raise ValueError("the batch must be sorted by date")
    out, i0 = [], 0
    for f in cum_fractions:
        # same rounding as the library (bp_upload_market_async: ceil(f * R))
        i1 = int(np.searchsorted(hi, int(np.ceil(f * n_hf_rows)), side="right"))
        if i1 > i0:
            out.append((i0, i1, slice_batch(batch, i0, i1)))
            i0 = i1
    if i0 < len(hi):
        out.append((i0, len(hi), slice_batch(batch, i0, len(hi))))
    return out


def trim_intraday(batch: WindowBatch):
    """Row range ``[lo, hi)`` of the intraday matrix that the windows of ``batch`` read; the batch is shifted in place
    so that it refers to ``hf_prices[lo:hi]``.  Bars outside the range (e.g. the years of history before the first
    rebalance date that only the DAILY windows need) are never touched by any window and need not be uploaded."""
    if batch.hf_lo is None or batch.hf_hi is None:
        raise ValueError("this batch has no intraday window rows")
    lo, hi = int(batch.hf_lo.min()), int(batch.hf_hi.max())
    batch.hf_lo = (batch.hf_lo - lo).astype(np.int32)
    batch.hf_hi = (batch.hf_hi - lo).astype(np.int32)
    return lo, hi


@dataclass
class ResampledRows:
    """Return rows of weekly windows, built on the device from the daily prices (``bp_set_resampled``):
    row i = ln(P[num_row[i]] / P[den_row[i]]).  Rows 0..n_weeks-1: week close against the previous week's close
    (``resample('W').last()``, :153); rows n_weeks..n_weeks+D-1: price at trading date d against the previous
    week's close (the partial last week of a window).  ``rf_row`` / ``mcm`` carry the risk-free rate forward-filled
    at each row's Sunday label (:54 — including the look-ahead of the partial week's label) and the MCM value."""
    num_row: np.ndarray
    den_row: np.ndarray
    rf_row: np.ndarray
    mcm: Optional[np.ndarray]
    n_weeks: int


def week_ids(dates: np.ndarray) -> np.ndarray:
    """Bucket of ``resample('W')`` (weeks end on Sunday; 1970-01-01 is a Thursday)."""
    return (dates.astype("datetime64[D]").astype(np.int64) + 3) // 7


def plan_weekly_windows(spec, dates: np.ndarray, d_indices: Sequence[int], rf_dates: np.ndarray, rf_values: np.ndarray,
                        mcm: Optional[np.ndarray] = None, hf_ts: Optional[np.ndarray] = None,
                        hf_lookback_days: Optional[int] = None, need_hf: bool = True):
    """Window descriptors for ``rolling_window_frequency == 'weekly'`` (:104-106, :151-153).

    A window at date d holds the closes of the n-1 complete weeks before d's week plus the price at d; its n-1
    returns are n-2 shared weekly rows and one per-date row.  Returns (ResampledRows, WindowBatch).
    """
    n = int(spec["rolling_window"])
    D = len(dates)
    wid = week_ids(dates)
    if np.any(np.diff(wid) > 1):
        raise NotImplementedError("empty week in resample('W'): the reference would emit a NaN row")
    wk = wid - wid[0]                                   # week index of every trading date
    n_weeks = int(wk[-1]) + 1
    last = np.r_[np.nonzero(np.diff(wk))[0], D - 1]     # last trading row of every week
    prev_close = np.where(wk >= 1, last[np.maximum(wk - 1, 0)], np.arange(D))
    num = np.r_[last, np.arange(D)].astype(np.int32)
    den = np.r_[np.r_[last[0], last[:-1]], prev_close].astype(np.int32)
    labels = ((wid[0] + np.arange(n_weeks)) * 7 + 3).astype("datetime64[D]").astype("datetime64[ns]")   # Sundays
    rf_week = ffill_rows(labels, rf_dates, rf_values)
    rf_row = np.r_[rf_week, rf_week[wk]]
    mcm_rows = None
    if mcm is not None:
        mcm = np.atleast_2d(np.asarray(mcm, dtype=np.float64))
        mcm_rows = np.concatenate([mcm[:, last], mcm], axis=1)
    rows = ResampledRows(num, den, rf_row.astype(np.float64), mcm_rows, n_weeks)

    d_idx = np.asarray(d_indices, dtype=np.int64)
    k = wk[d_idx]
    if k.min() < n - 1:
        raise ValueError(f"a weekly window of {n} prices needs {n - 1} complete weeks before the trade date")
    hf_lo = hf_hi = None
    if need_hf:
        if hf_ts is None:
            raise ValueError("intraday timestamps required for the conjugate prior")
        Dd = hf_lookback(spec, hf_lookback_days)
        dd = dates[d_idx]
        hf_lo = np.searchsorted(hf_ts, dd - Dd * _DAY + _DAY, side="right").astype(np.int32)
        hf_hi = np.searchsorted(hf_ts, dd + _DAY, side="right").astype(np.int32)
    strat = spec["weighting_strategy"]
    conj = strat.startswith("conjugate")
    batch = WindowBatch(
        rolling_window=n,
        day_row=(k - 1).astype(np.int32),                              # last shared weekly row
        span_days=np.full(len(d_idx), 7 * (n - 1), dtype=np.int32),    # labels are consecutive Sundays
        hf_lo=hf_lo, hf_hi=hf_hi,
        mcm_index=mcm_index_of(strat) if conj else 0,
        mcm_scaling=float(spec["mcm_scaling"]) if conj and spec.get("mcm_scaling") is not None else 1.0,
        risk_aversion=float(spec["risk_aversion"]) if spec.get("risk_aversion") is not None else 1.0,
        prior_weights=prior_kind_of(strat) if conj else 0,
        resampled=True,
        extra_row=(n_weeks + d_idx).astype(np.int32),
        caps_row=d_idx.astype(np.int32),
    )
    return rows, batch


@dataclass
class StackedWindows:
    """Windows laid out in one stacked working market (``BayesEngine.select_windows``): window w owns the daily pool
    rows [day_lo[w], day_hi[w]), which start at stack row day_off[w], and the intraday pool rows [hf_lo[w], hf_hi[w]) at
    stack row hf_off[w] (``None``: no intraday rows).  ``batch`` and, for weekly windows, ``resampled`` name stack rows."""
    batch: WindowBatch
    resampled: Optional[ResampledRows]
    day_lo: np.ndarray
    day_hi: np.ndarray
    day_off: np.ndarray
    hf_lo: Optional[np.ndarray]
    hf_hi: Optional[np.ndarray]
    hf_off: Optional[np.ndarray]


def _block_offsets(lengths: np.ndarray) -> np.ndarray:
    return np.r_[0, np.cumsum(lengths)[:-1]].astype(np.int64)


def stack_windows(batch: WindowBatch, rows: Optional[ResampledRows] = None) -> StackedWindows:
    """Relocate windows planned on the full calendar (``plan_daily_windows`` without row offsets, or
    ``plan_weekly_windows`` and its ``rows``) into one block each of a stacked market, in batch order.

    A block holds the rows a ``select_market`` slice gives the window, at the same positions relative to the window:
    daily windows the n prices up to the trade date; weekly windows the daily rows from the first week close their
    returns read up to the trade date (its caps row); intraday rows from one row in front of the window's first bar
    (``hf_lo - 1``, as the per-set slices keep it) to its last.  Weekly windows get their own copy of the resampled
    rows they read -- n-2 week rows then the trade date's row, each with its ``rf_row`` value (the partial week's
    look-ahead label included) and ``num_row`` / ``den_row`` moved into the block -- behind one unused row 0.  Nothing
    is re-derived, so every descriptor equals the plan's up to the block offsets."""
    W, n = batch.n_windows, int(batch.rolling_window)
    dr = batch.day_row.astype(np.int64)
    res = None
    if batch.resampled:
        if rows is None:
            raise ValueError("weekly windows need the ResampledRows of their plan")
        # resampled rows of every window: its n-2 shared week rows, then its own trade-date row
        sel = np.concatenate([dr[:, None] + np.arange(-(n - 3), 1)[None, :], batch.extra_row.astype(np.int64)[:, None]], axis=1)
        num, den = rows.num_row[sel].astype(np.int64), rows.den_row[sel].astype(np.int64)
        caps = batch.caps_row.astype(np.int64)
        day_lo = np.minimum(np.minimum(num.min(axis=1), den.min(axis=1)), caps)
        day_hi = np.maximum(np.maximum(num.max(axis=1), den.max(axis=1)), caps) + 1
        day_off = _block_offsets(day_hi - day_lo)
        shift = (day_off - day_lo)[:, None]
        mcm = None
        if rows.mcm is not None:
            mcm = np.concatenate([np.zeros((rows.mcm.shape[0], 1)), rows.mcm[:, sel.ravel()]], axis=1)
        res = ResampledRows(num_row=np.r_[0, (num + shift).ravel()].astype(np.int32),
                            den_row=np.r_[0, (den + shift).ravel()].astype(np.int32),
                            rf_row=np.r_[0.0, rows.rf_row[sel.ravel()]].astype(np.float64), mcm=mcm,
                            n_weeks=1 + W * (n - 1))
        first = 1 + np.arange(W, dtype=np.int64) * (n - 1)
        day_row, extra_row, caps_row = first + n - 3, first + n - 2, caps - day_lo + day_off
    else:
        day_lo, day_hi = dr - (n - 1), dr + 1
        if day_lo.min() < 0:
            raise ValueError(f"a window of {n} prices needs {n - 1} rows before the trade date")
        day_off = _block_offsets(day_hi - day_lo)
        day_row, extra_row = dr - day_lo + day_off, batch.extra_row
        caps_row = None if batch.caps_row is None else batch.caps_row - day_lo + day_off
    hf_lo = hf_hi = hf_off = new_lo = new_hi = None
    if batch.hf_lo is not None:
        lo, hf_hi = batch.hf_lo.astype(np.int64), batch.hf_hi.astype(np.int64)
        hf_lo = np.maximum(lo - 1, 0)
        hf_off = _block_offsets(hf_hi - hf_lo)
        new_lo, new_hi = lo - hf_lo + hf_off, hf_hi - hf_lo + hf_off
    i32 = lambda a: None if a is None else np.asarray(a).astype(np.int32)
    import dataclasses
    stacked = dataclasses.replace(batch, day_row=i32(day_row), hf_lo=i32(new_lo), hf_hi=i32(new_hi),
                                  extra_row=i32(extra_row), caps_row=i32(caps_row))
    return StackedWindows(stacked, res, day_lo, day_hi, day_off, hf_lo, hf_hi, hf_off)


def stack_batches(n_cols: Sequence[int], window_bytes: Sequence[int], budget: int):
    """Positions of the windows of each stacked batch: windows with the same number of columns (a stacked market has
    one N), in their given order, cut so that a batch's ``window_bytes`` stay within ``budget`` (a window larger than
    the budget forms a batch of its own)."""
    n_cols = np.asarray(n_cols, dtype=np.int64)
    out = []
    for N in dict.fromkeys(n_cols.tolist()):
        pos = np.nonzero(n_cols == N)[0]
        start, acc = 0, 0
        for k, i in enumerate(pos):
            b = int(window_bytes[i])
            if k > start and acc + b > budget:
                out.append(pos[start:k])
                start, acc = k, 0
            acc += b
        out.append(pos[start:])
    return out


def mcm_prior_n(spec, mcm_dates: np.ndarray, mcm_values: np.ndarray, trade_dates: np.ndarray) -> np.ndarray:
    """``calculate_conjugate_prior_n`` (:247-267) for many trade dates, on the MCM series' OWN calendar.

    The reference averages the last ``rolling_window`` observations of the MCM frame it is handed (rows <= d, :977-983),
    whatever their dates are — FRED's daily EPU index has 7 observations per week, VIX has 5 — and for weekly windows
    the last observation of every ``resample('W')`` bucket (:106), the bucket of d ending at d itself.  Empty buckets
    are NaN rows that ``iloc[-n:]`` counts and ``mean()`` skips.  A trade date missing from the MCM index raises the
    reference's ``ValueError`` (:98-100).  Returns ``n0`` [W], to be passed as ``WindowBatch.prior_n``."""
    n = int(spec["rolling_window"])
    freq = spec["rolling_window_frequency"]
    s = float(spec["mcm_scaling"])
    md = np.asarray(mcm_dates).astype("datetime64[ns]")
    mv = np.asarray(mcm_values, dtype=np.float64)
    order = np.argsort(md, kind="stable")                                   # sort_index() (:95)
    md, mv = md[order], mv[order]
    td = np.asarray(trade_dates).astype("datetime64[ns]")
    pos = np.searchsorted(md, td, side="right") - 1                          # last observation <= d
    bad = (pos < 0) | (md[np.maximum(pos, 0)] != td)
    if bad.any():
        d = td[np.nonzero(bad)[0][0]]
        raise ValueError(f"trading_date_ts {d} must be the last date in the DataFrame.")   # :98-100
    cur = mv[pos]                                                           # mcm_prices_df.loc[d] (:257)
    avg = np.empty(len(td))
    if freq == "daily":
        for i, p in enumerate(pos):
            avg[i] = np.nanmean(mv[max(0, p - n + 1): p + 1])              # iloc[-n:].mean() (:112)
    elif freq == "weekly":
        wid = week_ids(md)
        w0 = int(wid[0])
        n_weeks = int(wid[-1]) - w0 + 1
        week_last = np.full(n_weeks, np.nan)
        ok = ~np.isnan(mv)
        week_last[wid[ok] - w0] = mv[ok]                                    # last() = last non-NaN; ascending dates: the last write wins
        for i, p in enumerate(pos):
            k = int(wid[p]) - w0                                            # bucket of d ends at d (the frame is cut at d)
            j, own = int(p), np.nan
            while j >= 0 and wid[j] == wid[p]:
                if ok[j]:
                    own = mv[j]
                    break
                j -= 1
            vals = np.r_[week_last[max(0, k - n + 1): k], own]
            avg[i] = np.nanmean(vals)
    elif freq == "monthly":
        raise NotImplementedError("monthly windows: resample('M') was removed from pandas (SURVEY F10)")
    else:
        raise RuntimeError("Unknown rolling window frequency.")
    frac = np.where(cur > avg, cur / avg, avg / cur)                         # :260-263
    return n * frac * s                                                      # :265


def ffill_rows(target_dates: np.ndarray, src_dates: np.ndarray, src_values: np.ndarray) -> np.ndarray:
    """``series.reindex(target, method='ffill')`` (:54) for sorted date arrays."""
    idx = np.searchsorted(src_dates, target_dates, side="right") - 1
    out = np.where(idx >= 0, src_values[np.maximum(idx, 0)], np.nan)
    return out.astype(np.float64)


def cap_descending_order(caps_row: np.ndarray, size: int, eligible: Optional[np.ndarray] = None) -> np.ndarray:
    """Asset set and order of one window: ``nlargest(size)`` of the caps at d (:653-654, F7)."""
    cand = np.arange(caps_row.shape[0]) if eligible is None else np.asarray(eligible)
    return cand[np.argsort(-caps_row[cand], kind="stable")][:size]
