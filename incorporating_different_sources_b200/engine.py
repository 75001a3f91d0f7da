"""Batched Bayesian tangency-weight engine: the host side above the C-ABI.

``BayesEngine`` keeps one market resident in HBM and evaluates *all* rebalance windows of a
backtest per call (the reference evaluates one window per Python call,
``portfolio_calculations.py:1232-1234``).  PyTorch is used only as plumbing: device output
buffers, the CUDA stream, and (in ``sharding.py``) ``torch.distributed``.
"""
from __future__ import annotations

import ctypes as C
from typing import Dict, Iterable, Optional, Sequence

import numpy as np

from . import _lib
from ._lib import BP_NSCAL, SCAL, MarketDesc, Outputs, WindowBatchDesc
from .windows import WindowBatch

VEC_OUTPUTS = ("weights", "nu", "w1", "t", "w0", "rhs")
MAT_OUTPUTS = ("T", "S0", "S1")
ALL_OUTPUTS = VEC_OUTPUTS + MAT_OUTPUTS + ("scalars", "status")


class BayesPortfolioError(RuntimeError):
    pass


def _raise(rc: int):
    msg = _lib.last_error()
    if rc == _lib.BP_ERR_INVALID:
        raise ValueError(msg)
    raise BayesPortfolioError(f"libbayes_portfolio error {rc}: {msg}")


def _c64(a) -> np.ndarray:
    return np.ascontiguousarray(a, dtype=np.float64)


def _market_desc(prices, rf_row, caps, hf_prices):
    """The descriptor of a market or pool upload (no MCM series) and the coerced arrays it points into, which must stay
    alive as long as the library reads them."""
    prices = _c64(prices)
    rf_row = _c64(rf_row)
    D, N = prices.shape
    if rf_row.shape != (D,):
        raise ValueError("rf_row must have one entry per daily row")
    if np.isnan(rf_row).any():
        raise ValueError("risk-free rate undefined on some window dates (the reference would drop rows, :60)")
    desc = MarketDesc()                   # unset pointers are NULL, unset counts 0
    desc.n_assets, desc.n_days = N, D
    desc.prices, desc.rf_row = prices.ctypes.data, rf_row.ctypes.data
    keep = [prices, rf_row]
    if caps is not None:
        caps = _c64(caps)
        if caps.shape != (D, N):
            raise ValueError("caps must match prices")
        keep.append(caps)
        desc.caps = caps.ctypes.data
    if hf_prices is not None and len(hf_prices):
        hf_prices = _c64(hf_prices)
        if hf_prices.shape[1] != N:
            raise ValueError("hf_prices must have N columns")
        keep.append(hf_prices)
        desc.hf_prices = hf_prices.ctypes.data
        desc.n_hf_rows = hf_prices.shape[0]
    return desc, keep


class BayesEngine:
    """One CUDA device, one resident market.

    Parameters
    ----------
    device : CUDA device ordinal.
    use_torch_stream : launch on torch's current stream so that ``torch.cuda.Event`` timing and
        ``torch.distributed`` collectives order correctly with the kernels.
    """

    def __init__(self, device: int = 0, use_torch_stream: bool = True, stream=None):
        self._lib = _lib.load()
        h = C.c_void_p()
        rc = self._lib.bp_init(int(device), C.byref(h))
        if rc != 0:
            _raise(rc)
        self._h = h
        self.device = int(device)
        self.n_assets = 0
        self.n_days = 0
        self.n_hf_rows = 0
        self.condition_estimate = False
        self.reuse_min_windows = 32      # library defaults (bp_set_reuse_min_windows / bp_set_jeffreys_chain)
        self.jeffreys_chain = 8
        self._stack_max = 15
        self._torch = None
        self._stream = stream        # a torch.cuda.Stream of this engine's own (two engines then overlap on one GPU)
        if use_torch_stream or stream is not None:
            import torch
            self._torch = torch
            torch.cuda.set_device(self.device)
            self.bind_torch_stream()

    # ------------------------------------------------------------------ plumbing
    def bind_torch_stream(self):
        torch = self._torch
        stream = (self._stream if self._stream is not None else torch.cuda.current_stream(self.device)).cuda_stream
        rc = self._lib.bp_set_stream(self._h, C.c_void_p(stream))
        if rc:
            _raise(rc)

    def close(self):
        if getattr(self, "_h", None) is not None and self._h:
            self._lib.bp_destroy(self._h)
            self._h = None

    def __del__(self):  # pragma: no cover
        try:
            self.close()
        except Exception:
            pass

    def synchronize(self):
        rc = self._lib.bp_synchronize(self._h)
        if rc:
            _raise(rc)
        self._inflight = None

    def wait_upload(self):
        """Block until the intraday block of the last asynchronous ``upload_market`` has arrived in HBM."""
        rc = self._lib.bp_wait_upload(self._h)
        if rc:
            _raise(rc)

    def set_workspace_limit(self, nbytes: int):
        rc = self._lib.bp_set_workspace_limit(self._h, C.c_size_t(int(nbytes)))
        if rc:
            _raise(rc)

    def device_info(self) -> Dict[str, int]:
        sm = C.c_int()
        fr = C.c_size_t()
        tot = C.c_size_t()
        rc = self._lib.bp_device_info(self._h, C.byref(sm), C.byref(fr), C.byref(tot))
        if rc:
            _raise(rc)
        return {"sm_count": sm.value, "free_bytes": fr.value, "total_bytes": tot.value}

    def set_stage_timing(self, enable: bool):
        rc = self._lib.bp_set_stage_timing(self._h, int(bool(enable)))
        if rc:
            _raise(rc)

    def stage_times(self) -> Dict[str, Dict[str, float]]:
        """Summed CUDA-event milliseconds and launch counts per stage since the last call."""
        ms = (C.c_double * _lib.BP_NSTAGE)()
        cnt = (C.c_longlong * _lib.BP_NSTAGE)()
        rc = self._lib.bp_get_stage_times(self._h, ms, cnt)
        if rc:
            _raise(rc)
        return {name: {"ms": ms[i], "launches": int(cnt[i])} for i, name in enumerate(_lib.STAGES)}

    def gram_work(self) -> Dict[str, float]:
        """Work counters of the Gram stage since the last call (rows on the tensor cores, block tiles added...)."""
        out = (C.c_double * 4)()
        rc = self._lib.bp_get_gram_work(self._h, out)
        if rc:
            _raise(rc)
        return {"k_rows": out[0], "add_blocks": out[1], "precompute_rows": out[2], "full_rows": out[3]}

    def set_jeffreys_chain(self, group: int = 8):
        """Jeffreys batches of consecutive trade dates factorise only every ``group``-th window and solve the others
        relative to it (Woodbury, rank 2k+4; ``jeffreys_chain.cu``); 0 or 1 factorises every window."""
        rc = self._lib.bp_set_jeffreys_chain(self._h, int(group))
        if rc:
            _raise(rc)
        self.jeffreys_chain = int(group)

    def set_condition_estimate(self, enable: bool):
        """Every window the solver factorises also gets ``scalars[:, SCAL["anorm1"]]`` (1-norm of the factorised
        matrix) and ``scalars[:, SCAL["rcond"]]``, LAPACK ``dpocon``'s reciprocal 1-norm condition estimate from the
        window's own Cholesky factor (0 for a window with a non-zero status).  While it is on, the Jeffreys chain is
        not used (every window is factorised); every other output is unchanged.  Off by default."""
        rc = self._lib.bp_set_condition_estimate(self._h, int(bool(enable)))
        if rc:
            _raise(rc)
        self.condition_estimate = bool(enable)

    def solve_work(self) -> Dict[str, float]:
        """Windows factorised / solved relative to a base window since the last call."""
        out = (C.c_double * 2)()
        rc = self._lib.bp_get_solve_work(self._h, out)
        if rc:
            _raise(rc)
        return {"factored": out[0], "chained": out[1]}

    def set_reuse_min_windows(self, n: int):
        """Smallest batch for which overlapping windows share precomputed block Gram tiles (2**31-1 disables)."""
        rc = self._lib.bp_set_reuse_min_windows(self._h, int(n))
        if rc:
            _raise(rc)
        self.reuse_min_windows = int(n)

    def set_stack_max_windows(self, n: int = 15):
        """Backtests evaluate the windows of every asset set with at most ``n`` windows together, in stacked batches
        (:meth:`select_windows`), instead of one working market and one batched call per set; 0 never stacks.  The
        results are the same bits either way.  Sets large enough for a route that shares work between windows keep
        their own call: :attr:`stack_max_windows` stays below the engine's block-reuse minimum and below the 2 x
        group windows of the Jeffreys chain."""
        if int(n) < 0:
            raise ValueError("n must be >= 0")
        self._stack_max = int(n)

    @property
    def stack_max_windows(self) -> int:
        """The largest asset set (in windows) that a backtest stacks: :meth:`set_stack_max_windows` capped by the
        routes that share work between the windows of one set."""
        cap = min(self._stack_max, self.reuse_min_windows - 1)
        if self.jeffreys_chain >= 2:
            cap = min(cap, 2 * self.jeffreys_chain - 1)
        return max(cap, 0)

    def set_hf_presum_min_days(self, min_days: int = 8):
        """Windows whose intraday look-back covers at least ``min_days`` trading days add at most three pre-summed
        (scanned) day-block tiles instead of one tile per day; 0 disables."""
        rc = self._lib.bp_set_hf_presum_min_days(self._h, int(min_days))
        if rc:
            _raise(rc)

    def set_async_outputs(self, enable: bool):
        """Batched calls with page-locked HOST outputs (``into=``) return once queued; results are complete after
        ``synchronize()``.  The host can then plan the next batch while the GPU works on the previous one."""
        rc = self._lib.bp_set_async_outputs(self._h, int(bool(enable)))
        if rc:
            _raise(rc)

    def set_upload_pipeline(self, segments: int = 8, min_bytes: int = 256 << 20):
        """Segments of an asynchronous intraday upload (1 disables) and the smallest block that is segmented."""
        rc = self._lib.bp_set_upload_pipeline(self._h, int(segments), int(min_bytes))
        if rc:
            _raise(rc)

    def set_upload_fractions(self, cum_fractions=None):
        """Explicit cumulative row fractions of the segments of the next asynchronous intraday uploads (at most 8;
        ``None`` restores the geometric default)."""
        if cum_fractions is None or len(cum_fractions) == 0:
            rc = self._lib.bp_set_upload_fractions(self._h, 0, None)
        else:
            arr = (C.c_double * len(cum_fractions))(*[float(x) for x in cum_fractions])
            rc = self._lib.bp_set_upload_fractions(self._h, len(cum_fractions), arr)
        if rc:
            _raise(rc)

    def solve_wave_windows(self) -> int:
        """Windows the solver factorises concurrently (6 per SM)."""
        return int(self._lib.bp_solve_wave_windows(self._h))

    def plan_upload_fractions(self, batch: WindowBatch, n_hf_rows: int, max_segments: int = 8):
        """Segment boundaries for a date-sorted conjugate batch: whole solver waves of windows per segment, so that
        every segment is solved at full occupancy while the next one is on the bus and less than one wave is left
        when the copy ends.  Returns cumulative row fractions for :meth:`set_upload_fractions`."""
        from .windows import plan_wave_fractions
        return plan_wave_fractions(batch.hf_hi, n_hf_rows, self.solve_wave_windows(), max_segments)

    @property
    def launch_count(self) -> int:
        return int(self._lib.bp_launch_count(self._h))

    # ------------------------------------------------------------------ market
    def upload_market(self, prices, rf_row, caps=None, hf_prices=None, mcm=None, async_copy=False):
        """Host arrays -> HBM.  With ``async_copy=True`` the arrays must be page-locked and are kept
        alive by the engine until :meth:`synchronize`; the intraday block then overlaps with stages that
        do not read it (Jeffreys, daily statistics).  ``prices`` [D][N], ``rf_row`` [D] (risk-free rate forward-filled onto
        the daily rows), ``caps`` [D][N], ``hf_prices`` [R][N], ``mcm`` [n_mcm][D] (row 0 VIX, row 1 EPU).

        ``hf_prices`` may hold NaN (missing bars).  As the reference's ``dropna`` (:314), an intraday return row with a
        NaN in any column is dropped: a NaN bar removes the returns on both sides of it.  A conjugate window uses the
        m returns it keeps (scalar ``m``); with m < 2 its S0 and weights are NaN and its status is non-zero."""
        desc, keep = _market_desc(prices, rf_row, caps, hf_prices)
        if mcm is not None:
            mcm = _c64(mcm)
            if mcm.ndim == 1:
                mcm = mcm[None, :]
            if mcm.shape[1] != desc.n_days:
                raise ValueError("mcm series must be aligned with the daily rows")
            keep.append(mcm)
            desc.mcm = mcm.ctypes.data
            desc.n_mcm = mcm.shape[0]
        fn = self._lib.bp_upload_market_async if async_copy else self._lib.bp_upload_market
        rc = fn(self._h, C.byref(desc))
        if rc:
            _raise(rc)
        self.n_assets, self.n_days, self.n_hf_rows = desc.n_assets, desc.n_days, int(desc.n_hf_rows)
        self._inflight = keep if async_copy else None

    def upload_pool(self, prices, rf_row, caps=None, hf_prices=None):
        """The FULL market (every candidate column, every row) into a resident pool; :meth:`select_market` then builds
        the working market of a batch on the device.  ``upload_pool(None, None)`` releases the pool.  ``hf_prices`` may
        hold NaN as in :meth:`upload_market`; the rows to drop are decided on the selected columns only, so holes in
        columns a working market does not select change nothing."""
        if prices is None:
            rc = self._lib.bp_upload_pool(self._h, None)
            if rc:
                _raise(rc)
            self.pool_shape = None
            return
        desc, keep = _market_desc(prices, rf_row, caps, hf_prices)
        rc = self._lib.bp_upload_pool(self._h, C.byref(desc))
        del keep
        if rc:
            _raise(rc)
        self.pool_shape = (desc.n_days, desc.n_assets, int(desc.n_hf_rows))

    def select_market(self, cols, day_lo: int = 0, day_hi: Optional[int] = None, hf_lo: int = 0, hf_hi: Optional[int] = None):
        """Working market = pool columns ``cols`` (in that order), daily rows [day_lo, day_hi), intraday rows
        [hf_lo, hf_hi): gathered on the device.  Window rows of a following batch are relative to the slice
        (``plan_daily_windows(..., row_offset=day_lo, hf_row_offset=hf_lo)``)."""
        D, _, R = self.pool_shape
        cols = np.ascontiguousarray(cols, dtype=np.int32)
        sel = _lib.PoolSelect()
        sel.n_cols = int(cols.shape[0])
        sel.cols = cols.ctypes.data
        sel.day_lo, sel.day_hi = int(day_lo), int(D if day_hi is None else day_hi)
        sel.hf_lo, sel.hf_hi = int(hf_lo), int(R if hf_hi is None else hf_hi)
        rc = self._lib.bp_select_market(self._h, C.byref(sel))
        if rc:
            _raise(rc)
        self.n_assets, self.n_days, self.n_hf_rows = int(cols.shape[0]), sel.day_hi - sel.day_lo, int(sel.hf_hi - sel.hf_lo)

    def select_windows(self, cols_per_window, day_ranges, hf_ranges=None):
        """Stacked working market: window w gets its own block of pool rows -- daily rows ``day_ranges[w]`` = (lo, hi)
        and intraday rows ``hf_ranges[w]`` -- in its own pool columns ``cols_per_window[w]`` (one N for all), the
        blocks one after the other in window order.  A following batch names stack rows and each window must read its
        own block only (:func:`~.windows.stack_windows` plans both).  Every window is then evaluated exactly as on a
        :meth:`select_market` slice of its own; the routes that share work between windows are off until the next
        ``select_market`` / ``upload_market``.  Returns the blocks' first stack rows (daily, intraday)."""
        cols = np.ascontiguousarray(cols_per_window, dtype=np.int32)
        if cols.ndim != 2:
            raise ValueError("cols_per_window must be [W][N]")
        W = cols.shape[0]
        days = np.ascontiguousarray(day_ranges, dtype=np.int64).reshape(-1, 2)
        if days.shape[0] != W:
            raise ValueError("day_ranges must have one (lo, hi) per window")
        day_lo, day_hi = np.ascontiguousarray(days[:, 0], dtype=np.int32), np.ascontiguousarray(days[:, 1], dtype=np.int32)
        day_off = np.ascontiguousarray(np.r_[0, np.cumsum(days[:, 1] - days[:, 0])[:-1]], dtype=np.int32)
        sel = _lib.WindowSelect()
        sel.n_windows, sel.n_cols = W, int(cols.shape[1])
        sel.cols, sel.day_lo, sel.day_hi, sel.day_off = cols.ctypes.data, day_lo.ctypes.data, day_hi.ctypes.data, day_off.ctypes.data
        sel.hf_lo = sel.hf_hi = sel.hf_off = None
        hf_off = None
        n_hf = 0
        if hf_ranges is not None:
            hf = np.ascontiguousarray(hf_ranges, dtype=np.int64).reshape(-1, 2)
            if hf.shape[0] != W:
                raise ValueError("hf_ranges must have one (lo, hi) per window")
            hf_lo, hf_hi = np.ascontiguousarray(hf[:, 0]), np.ascontiguousarray(hf[:, 1])
            hf_off = np.ascontiguousarray(np.r_[0, np.cumsum(hf_hi - hf_lo)[:-1]], dtype=np.int64)
            sel.hf_lo, sel.hf_hi, sel.hf_off = hf_lo.ctypes.data, hf_hi.ctypes.data, hf_off.ctypes.data
            n_hf = int((hf_hi - hf_lo).sum())
        rc = self._lib.bp_select_windows(self._h, C.byref(sel))
        if rc:
            _raise(rc)
        self.n_assets, self.n_days, self.n_hf_rows = int(cols.shape[1]), int((days[:, 1] - days[:, 0]).sum()), n_hf
        return day_off.astype(np.int64), hf_off

    def set_resampled(self, rows):
        """Build the weekly return rows (:class:`~.windows.ResampledRows`) on the device from the resident prices."""
        num = np.ascontiguousarray(rows.num_row, dtype=np.int32)
        den = np.ascontiguousarray(rows.den_row, dtype=np.int32)
        rf = _c64(rows.rf_row)
        r = _lib.ResampledDesc()
        r.n_rows = int(num.shape[0])
        r.num_row, r.den_row, r.rf_row = num.ctypes.data, den.ctypes.data, rf.ctypes.data
        mcm = None
        r.mcm = None
        if rows.mcm is not None:
            mcm = _c64(rows.mcm)
            r.mcm = mcm.ctypes.data
        rc = self._lib.bp_set_resampled(self._h, C.byref(r))
        if rc:
            _raise(rc)

    def prepare_market(self):
        """Re-run the on-device log-return stage (used to time the whole device path)."""
        rc = self._lib.bp_prepare_market(self._h)
        if rc:
            _raise(rc)

    # ------------------------------------------------------------------ batches
    def _batch_desc(self, b: WindowBatch, need_hf: bool):
        keep = []
        d = WindowBatchDesc()
        d.n_windows = b.n_windows
        d.rolling_window = int(b.rolling_window)
        for name in ("day_row", "span_days"):
            a = np.ascontiguousarray(getattr(b, name), dtype=np.int32)
            keep.append(a)
            setattr(d, name, a.ctypes.data)
        d.hf_lo = None
        d.hf_hi = None
        if need_hf:
            if b.hf_lo is None or b.hf_hi is None:
                raise ValueError("this batch has no intraday window rows")
            for name in ("hf_lo", "hf_hi"):
                a = np.ascontiguousarray(getattr(b, name), dtype=np.int32)
                keep.append(a)
                setattr(d, name, a.ctypes.data)
        d.mcm_index = int(b.mcm_index)
        d.mcm_scaling = float(b.mcm_scaling)
        d.risk_aversion = float(b.risk_aversion)
        d.prior_weights = int(b.prior_weights)
        d.mcm_rows = int(getattr(b, "mcm_rows", 0) or 0)
        d.resampled = int(bool(getattr(b, "resampled", False)))
        d.extra_row = None
        d.caps_row = None
        if d.resampled:
            for name in ("extra_row", "caps_row"):
                a = np.ascontiguousarray(getattr(b, name), dtype=np.int32)
                keep.append(a)
                setattr(d, name, a.ctypes.data)
        d.prior_n = None
        if getattr(b, "prior_n", None) is not None:
            pn = np.ascontiguousarray(b.prior_n, dtype=np.float64)
            if pn.shape != (b.n_windows,):
                raise ValueError("prior_n must have one entry per window")
            keep.append(pn)
            d.prior_n = pn.ctypes.data
        return d, keep

    def _alloc_outputs(self, W: int, names: Iterable[str], device_out: bool, into: Optional[dict],
                       n_assets: Optional[int] = None):
        N = self.n_assets if n_assets is None else n_assets
        o = Outputs()
        res = {}
        for f, _ in Outputs._fields_:
            setattr(o, f, None)
        for name in names:
            if name not in ALL_OUTPUTS:
                raise KeyError(name)
            if name in VEC_OUTPUTS:
                shape, dt = (W, N), np.float64
            elif name in MAT_OUTPUTS:
                shape, dt = (W, N, N), np.float64
            elif name == "scalars":
                shape, dt = (W, BP_NSCAL), np.float64
            else:
                shape, dt = (W,), np.int32
            if into is not None and name in into:
                buf = into[name]
            elif device_out:
                torch = self._torch
                buf = torch.empty(shape, dtype=torch.float64 if dt is np.float64 else torch.int32,
                                  device=f"cuda:{self.device}")
            else:
                buf = np.empty(shape, dtype=dt)
            res[name] = buf
            ptr = buf.data_ptr() if hasattr(buf, "data_ptr") else buf.ctypes.data
            setattr(o, name, ptr)
        return o, res

    def _run(self, fn, b: WindowBatch, outputs, device_out, into, need_hf):
        d, keep = self._batch_desc(b, need_hf)
        o, res = self._alloc_outputs(b.n_windows, outputs, device_out, into)
        rc = fn(self._h, C.byref(d), C.byref(o))
        del keep
        if rc:
            _raise(rc)
        return res

    def conjugate(self, batch: WindowBatch, outputs: Sequence[str] = ("weights", "status"),
                  device_out: bool = False, into: Optional[dict] = None) -> Dict[str, object]:
        """``calculate_conjugate_hf_mcm_portfolio`` (:819-836) for every window of the batch."""
        return self._run(self._lib.bp_conjugate_batched, batch, outputs, device_out, into, True)

    def jeffreys(self, batch: WindowBatch, outputs: Sequence[str] = ("weights", "status"),
                 device_out: bool = False, into: Optional[dict] = None) -> Dict[str, object]:
        """``calculate_jeffreys_portfolio`` (:838-849) for every window of the batch."""
        return self._run(self._lib.bp_jeffreys_batched, batch, outputs, device_out, into, False)

    def _estimator(self, which: int, batch: WindowBatch, outputs, device_out, into):
        lib = self._lib

        def fn(h, d, o):
            return lib.bp_estimator_batched(h, d, which, o)
        return self._run(fn, batch, outputs, device_out, into, False)

    def jorion(self, batch: WindowBatch, outputs: Sequence[str] = ("weights", "status"),
               device_out: bool = False, into: Optional[dict] = None) -> Dict[str, object]:
        """``calculate_jorion_portfolio`` (:851-895) for every window of the batch: one factorisation of the
        centred Gram, two right-hand sides, Bayes-Stein combination in the solver's epilogue."""
        from ._lib import EST_JORION
        return self._estimator(EST_JORION, batch, outputs, device_out, into)

    def shrinkage(self, batch: WindowBatch, outputs: Sequence[str] = ("weights", "status"),
                  device_out: bool = False, into: Optional[dict] = None) -> Dict[str, object]:
        """``calculate_shrinkage_portfolio`` (:703-758) in closed form, ``(1/gamma) Sigma_LW^-1 mu_hat`` with the
        Ledoit-Wolf covariance (unrounded: the reference's ``clean_weights()`` rounding is the facade's job).  With s
        the shrinkage intensity (``scalars[:, SCAL_LW["shrinkage"]]``), ``S1`` is ``m Sigma_LW / (1 - s)`` and ``rhs``
        ``t / (1 - s)``, m = rolling_window - 1.  As in sklearn, s = 0 for one asset, and a window whose intensity
        clips (s = 1 exactly) has Sigma_LW = mu I: its ``S1`` is ``m Sigma_LW = mu m I`` and its ``rhs`` is ``t``."""
        from ._lib import EST_SHRINKAGE
        return self._estimator(EST_SHRINKAGE, batch, outputs, device_out, into)

    def moments(self, batch: WindowBatch, outputs: Sequence[str], jeffreys: bool = False,
                device_out: bool = False, into: Optional[dict] = None) -> Dict[str, object]:
        """Posterior moments without the solve (t, w0, rhs, scalars, T, S0, S1)."""
        lib = self._lib

        def fn(h, d, o):
            return lib.bp_moments_batched(h, d, 1 if jeffreys else 0, o)
        return self._run(fn, batch, outputs, device_out, into, not jeffreys)

    def stats(self, batch: WindowBatch, want_T: bool = True):
        """``calculate_canonical_statistics_t`` / ``_T`` (:163-245)."""
        d, keep = self._batch_desc(batch, False)
        W, N = batch.n_windows, self.n_assets
        t = np.empty((W, N))
        T = np.empty((W, N, N)) if want_T else None
        rc = self._lib.bp_stats_batched(self._h, C.byref(d), t.ctypes.data, T.ctypes.data if want_T else None)
        del keep
        if rc:
            _raise(rc)
        return t, T

    def hf_cov(self, batch: WindowBatch):
        """``calculate_conjugate_prior_n`` / ``_S`` (:247-267, :285-333): (n0 [W], S0 [W][N][N])."""
        d, keep = self._batch_desc(batch, True)
        W, N = batch.n_windows, self.n_assets
        n0 = np.empty(W)
        S0 = np.empty((W, N, N))
        rc = self._lib.bp_hf_cov_batched(self._h, C.byref(d), n0.ctypes.data, S0.ctypes.data)
        del keep
        if rc:
            _raise(rc)
        return n0, S0


    # ------------------------------------------------------------------ loop body
    def backtest_loop(self, reb_rows, weights, distance_scale: float, turnover_cost_bps: float, member=None,
                      last_row: Optional[int] = None, device_out: bool = False):
        """Loop body of ``Portfolio.update_portfolio`` (:1127-1219) for a whole backtest.

        ``reb_rows`` [R] daily rows of the rebalance dates, ``weights`` [R][N] (NumPy, or a CUDA torch tensor
        as returned by ``conjugate(..., device_out=True)``).  Returns (returns [T], turnover [R-1], metrics [R][5]),
        NumPy arrays or, with ``device_out``, CUDA tensors (no device -> host copy).
        """
        reb = np.ascontiguousarray(reb_rows, dtype=np.int32)
        R = int(reb.shape[0])
        N = self.n_assets
        keep = [reb]
        if hasattr(weights, "data_ptr"):
            if tuple(weights.shape) != (R, N) or not weights.is_contiguous():
                raise ValueError("weights must be a contiguous [R][N] tensor")
            wptr = weights.data_ptr()
        else:
            w = _c64(weights)
            if w.shape != (R, N):
                raise ValueError("weights must be [R][N]")
            keep.append(w)
            wptr = w.ctypes.data
        d = _lib.BacktestDesc()
        d.n_rebalances = R
        d.reb_row = reb.ctypes.data
        last_row = int(reb[-1]) if last_row is None else int(last_row)
        d.last_row = last_row
        d.weights = wptr
        d.member = None
        if member is not None:
            m = np.ascontiguousarray(member, dtype=np.uint8)
            if m.shape != (R, N):
                raise ValueError("member must be [R][N]")
            keep.append(m)
            d.member = m.ctypes.data
        d.distance_scale = float(distance_scale)
        d.turnover_cost_bps = float(turnover_cost_bps)
        T = int(last_row - reb[0]) if R else 0
        if device_out:
            torch = self._torch
            dev = f"cuda:{self.device}"
            rets = torch.empty(max(T, 1), dtype=torch.float64, device=dev)[:max(T, 0)]
            to = torch.empty(max(R - 1, 1), dtype=torch.float64, device=dev)[:max(R - 1, 0)]
            met = torch.empty((R, 5), dtype=torch.float64, device=dev)
            d.returns, d.turnover, d.metrics = rets.data_ptr(), to.data_ptr(), met.data_ptr()
        else:
            rets = np.empty(max(T, 0))
            to = np.empty(max(R - 1, 0))
            met = np.empty((R, 5))
            d.returns, d.turnover, d.metrics = rets.ctypes.data, to.ctypes.data, met.ctypes.data
        rc = self._lib.bp_backtest_batched(self._h, C.byref(d))
        del keep
        if rc:
            _raise(rc)
        return rets, to, met

    # ------------------------------------------------------------------ single-window building blocks
    def excess_returns(self, batch: WindowBatch) -> np.ndarray:
        """``calculate_excess_log_returns_from_prices`` (:31-62) of a one-window batch."""
        d, keep = self._batch_desc(batch, False)
        X = np.empty((batch.rolling_window - 1, self.n_assets))
        rc = self._lib.bp_excess_returns(self._h, C.byref(d), X.ctypes.data)
        del keep
        if rc:
            _raise(rc)
        return X

    def quadratic_form(self, w: np.ndarray, S: np.ndarray) -> float:
        """``calculate_portfolio_variance`` (:64-88): w'Sw."""
        w = _c64(w)
        S = _c64(S)
        out = np.empty(1)
        rc = self._lib.bp_quadratic_form(self._h, int(w.shape[0]), w.ctypes.data, S.ctypes.data, out.ctypes.data)
        if rc:
            _raise(rc)
        return float(out[0])

    def dense_posterior(self, *, jeffreys: bool, rolling_window: int, risk_aversion: float, T, t, S0=None, w0=None,
                        n0: float = 0.0, n1=None, c=None, S1=None, w1=None) -> Dict[str, object]:
        """Posterior from dense (possibly injected) moments: the optional-argument forms of :382-608."""
        keep = []
        pr = _lib.DenseProblem()
        if T is None:
            N = int(np.asarray(w0).shape[0])
            pr.T = pr.t = None
        else:
            T = _c64(T)
            t = _c64(t)
            N = T.shape[0]
            keep += [T, t]
            pr.T, pr.t = T.ctypes.data, t.ctypes.data
        pr.n_assets, pr.jeffreys, pr.rolling_window = N, int(bool(jeffreys)), int(rolling_window)
        pr.risk_aversion = float(risk_aversion)
        pr.n0 = float(n0)
        for name, val, shape in (("S0", S0, (N, N)), ("w0", w0, (N,)), ("S1", S1, (N, N)), ("w1", w1, (N,))):
            if val is None:
                setattr(pr, name, None)
                continue
            a = _c64(val)
            if a.shape != shape:
                raise ValueError(f"{name} has shape {a.shape}, expected {shape}")
            keep.append(a)
            setattr(pr, name, a.ctypes.data)
        for name, val in (("n1", n1), ("c", c)):
            if val is None:
                setattr(pr, name, None)
            else:
                a = np.array([float(val)])
                keep.append(a)
                setattr(pr, name, a.ctypes.data)
        res = {"scalars": np.zeros(BP_NSCAL), "S1": np.empty((N, N)), "w1": np.empty(N), "nu": np.empty(N),
               "weights": np.empty(N), "status": np.zeros(1, dtype=np.int32)}
        out = _lib.DenseResult()
        for k, v in res.items():
            setattr(out, k, v.ctypes.data)
        rc = self._lib.bp_dense_posterior(self._h, C.byref(pr), C.byref(out))
        del keep
        if rc:
            _raise(rc)
        return res

    def solve(self, S, rhs, *, jeffreys: bool = True, n1=None, jorion: bool = False, n_returns: int = 0,
              risk_aversion: float = 1.0, outputs: Sequence[str] = ("weights", "nu", "w1", "scalars", "status"),
              ) -> Dict[str, np.ndarray]:
        """The solve stage alone on caller-supplied matrices ``S`` [W][N][N] (lower triangle read) and ``rhs`` [W][N]:
        ``w1 = S^-1 rhs``, ``v1 = w1'S w1`` and the epilogue of the conjugate (``n1`` [W], :485-489, :572-575), Jeffreys
        (:600-606) or, with ``jorion=True``, Jorion (``S`` = C, ``rhs`` = t, ``n_returns`` = m, :851-895) path."""
        S = _c64(S)
        rhs = _c64(rhs)
        if S.ndim != 3 or S.shape[1] != S.shape[2]:
            raise ValueError("S must be [W][N][N]")
        W, N = S.shape[0], S.shape[1]
        if rhs.shape != (W, N):
            raise ValueError(f"rhs has shape {rhs.shape}, expected {(W, N)}")
        d = _lib.SolveDesc()
        d.n_windows, d.n_assets = W, N
        d.jeffreys, d.estimator = int(bool(jeffreys)), _lib.EST_JORION if jorion else 0
        d.n_returns, d.risk_aversion = int(n_returns), float(risk_aversion)
        d.S, d.rhs = S.ctypes.data, rhs.ctypes.data
        keep = [S, rhs]
        d.n1 = None
        if n1 is not None:
            n1 = _c64(n1)
            if n1.shape != (W,):
                raise ValueError("n1 must have one entry per window")
            keep.append(n1)
            d.n1 = n1.ctypes.data
        o, res = self._alloc_outputs(W, outputs, False, None, n_assets=N)
        rc = self._lib.bp_solve_batched(self._h, C.byref(d), C.byref(o))
        del keep
        if rc:
            _raise(rc)
        return res


def scalars_to_dict(scal_row: np.ndarray) -> Dict[str, float]:
    return {k: float(scal_row[i]) for k, i in SCAL.items()}


def upload_synthetic(engine: BayesEngine, mkt, cols=None, day_slice: Optional[slice] = None):
    """Upload a :class:`SyntheticMarket` (optionally a column subset / contiguous day range).

    Returns (row_offset, hf_row_offset): what to subtract from market row numbers to obtain rows of
    the resident slice.
    """
    from .windows import ffill_rows
    cols = np.arange(mkt.n_assets) if cols is None else np.asarray(cols)
    ds = day_slice or slice(0, mkt.n_days)
    d0, d1 = ds.start or 0, ds.stop if ds.stop is not None else mkt.n_days
    bars = len(mkt.hf_ts) // mkt.n_days
    h0, h1 = d0 * bars, d1 * bars
    full = cols.shape[0] == mkt.n_assets and np.array_equal(cols, np.arange(mkt.n_assets))
    pick = (lambda a: a) if full else (lambda a: a[:, cols])
    rf_dates = getattr(mkt, "rf_dates", mkt.dates)
    rf_row = ffill_rows(mkt.dates[d0:d1], rf_dates, mkt.rf)
    engine.upload_market(
        prices=pick(mkt.prices[d0:d1]), rf_row=rf_row, caps=pick(mkt.caps[d0:d1]),
        hf_prices=pick(mkt.hf_prices[h0:h1]), mcm=np.stack([mkt.vix[d0:d1], mkt.epu[d0:d1]]))
    return d0, h0
