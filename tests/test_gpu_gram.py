"""The Gram stage on its own: T, S0, S1, J, Jorion's C, t, rhs and the moment scalars of every window, entry by entry
against the extended-precision reference of tests/_gram_ref.py and its a-priori bound, on every route the host plan
can pick (from scratch, daily block grids, intraday block grid, day blocks with gathered overnight rows, pre-summed
day blocks, pipelined, chunked, weekly) and at the tile / padding edges.  Each case asserts from the library's work
counters that it really took the route it names.  Where two routes run the same kernels on the same plan (chunked
and unchunked, pipelined and blocking) the results are compared bit for bit."""
import dataclasses

import numpy as np
import pytest

from oracle import bayes_oracle as bo
from tests import _gram_ref as gr
from tests._dropna_ref import use_dropna_oracle

pytestmark = pytest.mark.gpu

U = gr.U
NO_REUSE = 2 ** 31 - 1
CONJ_OUTS = ("T", "S0", "S1", "t", "w0", "rhs", "scalars")
JEFF_OUTS = ("T", "S1", "t", "scalars")
SC = dict(n0=0, alpha=2, beta=3, c=4, v0=5, m=6)
WORST = {}                 # route -> output -> worst |E| / bound seen (printed at the end of the module)


@pytest.fixture(scope="module")
def engine():
    from incorporating_different_sources_b200.engine import BayesEngine
    gr.require_extended_precision()
    eng = BayesEngine(0)
    yield eng
    eng.close()
    if WORST:
        print("\nworst |E| / bound per route:")
        for route, d in WORST.items():
            print(f"  {route:28s} " + " ".join(f"{k}={v:.3g}" for k, v in sorted(d.items())))


@pytest.fixture(autouse=True)
def dropna_oracle(monkeypatch):
    use_dropna_oracle(monkeypatch)


@dataclasses.dataclass
class Market:
    prices: np.ndarray
    rf_row: np.ndarray
    caps: np.ndarray
    hf_prices: np.ndarray
    mcm: np.ndarray
    dates: np.ndarray
    hf_ts: np.ndarray
    rf: np.ndarray
    vix: np.ndarray
    epu: np.ndarray

    @property
    def N(self):
        return self.prices.shape[1]

    def arrays(self):
        return dict(prices=self.prices, rf_row=self.rf_row, caps=self.caps, hf_prices=self.hf_prices, mcm=self.mcm)

    def columns(self, cols):
        return dataclasses.replace(self, prices=np.ascontiguousarray(self.prices[:, cols]),
                                   caps=np.ascontiguousarray(self.caps[:, cols]),
                                   hf_prices=np.ascontiguousarray(self.hf_prices[:, cols]))


def _market(N, D, seed, bars=78, irregular=False):
    from incorporating_different_sources_b200.synthetic import generate_market
    from incorporating_different_sources_b200.windows import ffill_rows
    s = generate_market(N, D, seed=seed, bars_per_day=bars)
    if irregular:           # half days, bars absent from the calendar, a day cut down to 9 bars (test_gpu_configs.py)
        rng = np.random.default_rng(seed)
        keep = np.ones(len(s.hf_ts), dtype=bool)
        for day in rng.choice(D, size=12, replace=False):
            keep[day * bars + bars // 2:(day + 1) * bars] = False
        keep[rng.choice(len(keep), size=60, replace=False)] = False
        keep[(D - 20) * bars + 9:(D - 19) * bars] = False
        s = dataclasses.replace(s, hf_ts=s.hf_ts[keep], hf_prices=np.ascontiguousarray(s.hf_prices[keep]))
    return Market(s.prices, ffill_rows(s.dates, s.dates, s.rf), s.caps, s.hf_prices, np.stack([s.vix, s.epu]),
                  s.dates, s.hf_ts, s.rf, s.vix, s.epu)


def _with_holes(mkt, batch, rng, n_iso=80):
    """NaN bars inside the rows the batch reads: isolated ones and at hf_lo / hf_hi - 1 of some windows."""
    H = mkt.hf_prices.copy()
    lo, hi = int(batch.hf_lo.min()), int(batch.hf_hi.max())
    for r, c in zip(rng.integers(lo, hi, n_iso), rng.integers(0, mkt.N, n_iso)):
        H[r, c] = np.nan
    for i in range(0, batch.n_windows, 4):
        H[batch.hf_lo[i], (2 * i) % mkt.N] = np.nan
        H[batch.hf_hi[i] - 1, (3 * i + 1) % mkt.N] = np.nan
    return dataclasses.replace(mkt, hf_prices=H)


def _spec(N, rw, strategy="conjugate_hf_vix_vw", freq="daily"):
    return dict(weighting_strategy=strategy, size=N, risk_aversion=5, turnover_cost=15, rebalancing_frequency="daily",
                rolling_window=rw, rolling_window_frequency=freq, mcm_scaling=1, display_name="x")


def _plan(mkt, spec, d_idx, look=1, need_hf=True):
    from incorporating_different_sources_b200.windows import plan_daily_windows
    return plan_daily_windows(spec, mkt.dates, d_idx, mkt.hf_ts, hf_lookback_days=look, need_hf=need_hf)


def _record(route, name, r):
    d = WORST.setdefault(route, {})
    d[name] = max(d.get(name, 0.0), r)


def _assert_ratio(route, name, r, i):
    _record(route, name, r)
    assert r < 1.0, f"{route}: {name} of window {i} is {r:.3g} x its bound"


def _symmetric(got):
    for k in ("T", "S0", "S1"):
        if k in got:
            assert np.array_equal(got[k], np.swapaxes(got[k], 1, 2)), f"{k} is not exactly symmetric"


def _cols_for(N, rows, rng):
    """A column subset when a full longdouble product of N x rows x N would dominate the test's time."""
    return gr.edge_columns(N, rng) if N * N * rows > 4e8 else None


def check_windows(route, engine, mkt, batch, got, windows, *, conjugate=True, jeffreys=False, jorion=False,
                  weekly_rows=None, spec=None, seed=0):
    """Hold every requested output of the listed windows to the bound."""
    from incorporating_different_sources_b200.windows import slice_batch
    _symmetric(got)
    rng = np.random.default_rng(seed)
    n = batch.rolling_window
    for i in windows:
        if weekly_rows is None:
            X = engine.excess_returns(slice_batch(batch, i, i + 1))
            a = gr.daily_adjustments(mkt.rf_row, gr.daily_return_rows(int(batch.day_row[i]), n), int(batch.span_days[i]))
        else:
            X, a = weekly_rows[i]
        H = gr.intraday_rows(mkt.hf_prices, int(batch.hf_lo[i]), int(batch.hf_hi[i])) if conjugate else None
        rows = X.shape[0] + (H.shape[0] if H is not None else 0)
        cols = _cols_for(mkt.N, rows, rng)
        T, t = gr.daily_ref(X, a, cols)
        if "t" in got:
            _assert_ratio(route, "t", gr.lower_ratio(got["t"][i], t), i)
        if "T" in got:
            _assert_ratio(route, "T", gr.lower_ratio(got["T"][i], T), i)
        if jeffreys or jorion:
            C = gr.centred_ref(T, t, n - 1 if jorion else n)
            if "S1" in got:
                _assert_ratio(route, "C" if jorion else "J", gr.lower_ratio(got["S1"][i], C), i)
            continue
        if not conjugate:
            continue
        s = got["scalars"][i]
        m = H.shape[0]
        assert s[SC["m"]] == m, (i, s[SC["m"]], m)
        n0, alpha = float(s[SC["n0"]]), float(s[SC["alpha"]])
        assert abs(alpha - n0 * m / (m - 1)) <= 4 * U * alpha, i
        assert s[SC["beta"]] == alpha * m
        if spec is not None:                       # n0 = n * frac of a mean over the MCM window (:247-267)
            d = mkt.dates[batch.day_row[i]]
            series = mkt.vix if "vix" in spec["weighting_strategy"] else mkt.epu
            ref_n0 = bo.conjugate_prior_n(spec, mkt.dates[:batch.day_row[i] + 1], series[:batch.day_row[i] + 1], d)
            assert abs(n0 - ref_n0) <= (n + 8) * U * ref_n0, i
        S0 = gr.s0_ref(H, alpha, cols)
        if "S0" in got:
            _assert_ratio(route, "S0", gr.lower_ratio(got["S0"][i], S0), i)
        if "S1" in got:
            _assert_ratio(route, "S1", gr.lower_ratio(got["S1"][i], gr.sum_ref(S0, T)), i)
        if cols is None and ("rhs" in got or s[SC["v0"]] != 0):
            w0 = got["w0"][i] if "w0" in got else None
            if w0 is None:
                caps = mkt.caps[batch.day_row[i]] if weekly_rows is None else mkt.caps[batch.caps_row[i]]
                w0 = caps / caps.sum()
            _, v0, (c, c_err), (rhs, rhs_err) = gr.moments_ref(S0, t, w0, n0)
            _assert_ratio(route, "v0", gr.scalar_ratio(s[SC["v0"]], v0.value, float(v0.bound(gr.C_VEC))), i)
            _assert_ratio(route, "c", gr.scalar_ratio(s[SC["c"]], c, c_err), i)
            if "rhs" in got:
                r = np.abs(got["rhs"][i].astype(np.longdouble) - rhs).astype(np.float64) / rhs_err
                _assert_ratio(route, "rhs", float(r.max()), i)


def _work_delta(engine, fn):
    engine.gram_work()
    l0 = engine.launch_count
    out = fn()
    return out, engine.gram_work(), engine.launch_count - l0


class knobs:
    """Set engine knobs for one block and restore the defaults afterwards."""

    def __init__(self, engine, reuse=None, presum=None, limit=None):
        self.e, self.reuse, self.presum, self.limit = engine, reuse, presum, limit

    def __enter__(self):
        if self.reuse is not None:
            self.e.set_reuse_min_windows(self.reuse)
        if self.presum is not None:
            self.e.set_hf_presum_min_days(self.presum)
        if self.limit is not None:
            self.e.set_workspace_limit(self.limit)

    def __exit__(self, *exc):
        self.e.set_reuse_min_windows(32)
        self.e.set_hf_presum_min_days(8)
        self.e.set_workspace_limit(24 << 30)


def _per_window(N, max_m):
    """batch_plan.cu make_layout without the pre-summed mat-vec partials (the chunked test asserts the chunk count it
    implies, so a change of the layout fails there rather than silently testing something else)."""
    ld, ldS = -(-N // 16) * 16, -(-N // 32) * 32
    return 8 * ((ldS + 8) * ldS + 9 * ld + 12 + max(max_m, 2) + (max_m & 1)) + 16


def _r8(r):
    return (r + 7) // 8 * 8


def _daily_grid_work(batch, B, F):
    """(k_rows, precompute_rows) of a daily-only batch on the coarse / fine block grid B / F (batch_plan.cu split_rows
    and its work counters); B = F = 0: from scratch."""
    K = batch.rolling_window - 1
    k_rows, c_rng, f_rng = 0, [], []
    for dr in batch.day_row:
        r0 = int(dr) - K + 1
        r1 = r0 + K
        if B == 0:
            k_rows += _r8(K)
            continue
        c_lo, c_hi = -(-r0 // B), r1 // B
        f_lo, f_hi = -(-r0 // F), r1 // F
        if c_hi > c_lo:
            c_rng += [c_lo, c_hi]
            f_rng += [f_lo, c_lo * B // F] if c_lo * B // F > f_lo else []
            f_rng += [c_hi * B // F, f_hi] if f_hi > c_hi * B // F else []
            k_rows += _r8(f_lo * F - r0) + _r8(r1 - f_hi * F)
        elif f_hi > f_lo:
            f_rng += [f_lo, f_hi]
            k_rows += _r8(f_lo * F - r0) + _r8(r1 - f_hi * F)
        else:
            k_rows += _r8(K)
    pre = sum((max(rg) - min(rg)) * _r8(size) for rg, size in ((c_rng, B), (f_rng, F)) if rg)
    return k_rows, pre


def _day_block_starts(lo, hi):
    """batch_plan.cu day_block_starts: every hf_lo / hf_hi, long stretches cut to the typical block length."""
    st = np.unique(np.r_[lo, hi]).astype(np.int64)
    if len(st) < 3:
        return st
    gaps = np.diff(st)
    typical = max(8, int(np.sort(gaps)[len(gaps) // 2]))
    cut = []
    for k in range(len(st) - 1):
        cut.append(int(st[k]))
        gap = int(st[k + 1] - st[k])
        if gap > 2 * typical:
            pieces = gap // typical
            cut += [int(st[k]) + gap * q // pieces for q in range(1, pieces)]
    cut.append(int(st[-1]))
    return np.array(cut)


def _presum_chunks(batch):
    """Chunks of pre-summed day blocks each window's run touches (batch_plan.cu gram_job: chunk = minL days; 1, 2 or 3,
    which is also the number of scanned tiles the window adds)."""
    st = _day_block_starts(batch.hf_lo, batch.hf_hi)
    c_lo = np.searchsorted(st, batch.hf_lo)
    c_hi = np.searchsorted(st, batch.hf_hi)
    C = int((c_hi - c_lo).min()) - 1
    nb = int(c_hi.max() - c_lo.min())
    lo = c_lo - c_lo.min()
    last = c_hi - c_lo.min() - 1
    qa = lo // C
    return np.where(np.minimum((qa + 1) * C, nb) > last, 1, np.where(last // C == qa + 2, 3, 2))


# ------------------------------------------------------------------------------------------------- device rows
def test_device_excess_returns_match_the_oracle(engine):
    """The daily rows the reference contracts are the device's own; they are the oracle's rows to a few ulp.  x = l - a:
    the log return l = log(P_r / P_r-1) of the same correctly rounded ratio is held to a few ulp of |x| and |l|, the
    risk-free adjustment a_k = (1 + rf)^e - 1 (the same in every column of a row, so it is read off the row) to a few ulp
    of 1 + a_k -- its rounding is that of a power close to 1, on the device and in NumPy alike."""
    from incorporating_different_sources_b200.windows import slice_batch
    N, n = 33, 60
    mkt = _market(N, 120, seed=1)
    engine.upload_market(**mkt.arrays())
    spec = _spec(N, n)
    d_idx = (70, 95, 119)
    batch = _plan(mkt, spec, list(d_idx), need_hf=False)
    for i, d in enumerate(d_idx):
        X = engine.excess_returns(slice_batch(batch, i, i + 1))
        _, _, Xo = bo.daily_statistics(spec, mkt, d, np.arange(N))
        rows = gr.daily_return_rows(d, n)
        lo = np.log(mkt.prices[rows] / mkt.prices[rows - 1])
        ao = lo[:, :1] - Xo[:, :1]
        a_dev = np.median(lo - X, axis=1, keepdims=True)           # the device's a_k, to rounding of x and l
        assert np.all(np.abs(a_dev - ao) <= 4 * np.spacing(1.0 + np.abs(ao)))
        assert np.all(np.abs(X - (lo - a_dev)) <= 4 * U * (np.abs(X) + np.abs(lo)))


# ------------------------------------------------------------------------------------------------- shape sweep
@pytest.mark.parametrize("N", [1, 2, 15, 16, 17, 31, 33, 127, 128, 129, 255, 256, 257, 500, 520])
def test_shapes_from_scratch(engine, N):
    """ld padding to 16 and the 128-column tiles: every entry of T, S0, S1 = S0 + T, J and the moments."""
    mkt = _market(N, 75, seed=100 + N)
    engine.upload_market(**mkt.arrays())
    spec = _spec(N, 60)
    d_idx = [71, 73, 74]
    batch = _plan(mkt, spec, d_idx)
    with knobs(engine, reuse=NO_REUSE):
        got, work, _ = _work_delta(engine, lambda: engine.moments(batch, outputs=CONJ_OUTS))
        jg, jwork, _ = _work_delta(engine, lambda: engine.moments(batch, outputs=JEFF_OUTS, jeffreys=True))
    assert work["add_blocks"] == 0 and jwork["add_blocks"] == 0
    check_windows(f"scratch N={N}", engine, mkt, batch, got, range(3), spec=spec, seed=N)
    check_windows(f"scratch N={N}", engine, mkt, batch, jg, range(3), conjugate=False, jeffreys=True, seed=N)


@pytest.mark.parametrize("K", [2, 31, 32, 33, 64, 251])
def test_daily_rows_from_scratch(engine, K):
    """K at the 32-row k-tile edge: the last k-tile of a window runs compute_tile<MASK> with 1..31 valid rows."""
    N = 40
    mkt = _market(N, K + 10, seed=200 + K)
    engine.upload_market(**mkt.arrays())
    spec = _spec(N, K + 1)
    batch = _plan(mkt, spec, [K + 7, K + 8, K + 9])
    with knobs(engine, reuse=NO_REUSE):
        got, work, _ = _work_delta(engine, lambda: engine.moments(batch, outputs=CONJ_OUTS))
        jg = engine.moments(batch, outputs=JEFF_OUTS, jeffreys=True)
    assert work["add_blocks"] == 0
    check_windows(f"scratch K={K}", engine, mkt, batch, got, range(3), spec=spec)
    check_windows(f"scratch K={K}", engine, mkt, batch, jg, range(3), conjugate=False, jeffreys=True)


@pytest.mark.parametrize("m", [31, 32, 33])
def test_intraday_rows_at_the_k_tile_edge(engine, m):
    N = 40
    mkt = _market(N, 70, seed=300 + m)
    engine.upload_market(**mkt.arrays())
    spec = _spec(N, 60)
    batch = _plan(mkt, spec, [66, 67, 68, 69])
    batch.hf_lo = (batch.hf_hi - m - 1).astype(np.int32)
    with knobs(engine, reuse=NO_REUSE):
        got = engine.moments(batch, outputs=CONJ_OUTS)
    assert np.all(got["scalars"][:, SC["m"]] == m)
    check_windows(f"scratch m={m}", engine, mkt, batch, got, range(4), spec=spec)


# ------------------------------------------------------------------------------------------------- daily grid
GRIDS = {"none": (0, 0), "64/16": (64, 16), "128/32": (128, 32)}


@pytest.mark.parametrize("W,K,gaps,grid", [(31, 128, False, "none"), (32, 128, False, "64/16"), (32, 127, False, "none"),
                                           (32, 511, False, "64/16"), (32, 512, False, "128/32"),
                                           (40, 251, True, "64/16")])
def test_daily_block_grid(engine, W, K, gaps, grid):
    """reuse_min_windows = 32 and the grid choice at K = 128 (64/16) and K = 512 (128/32): the rows on the tensor cores
    and the rows of the block precompute are those of the expected grid and of no other.  Sorted dates at most two rows
    apart run the banded prep; the same batch in reverse order does not (one launch fewer, the same plan)."""
    N = 64
    D = K + 2 * W + 4
    mkt = _market(N, D, seed=400 + K + W, bars=2)
    engine.upload_market(**mkt.arrays())
    spec = _spec(N, K + 1, strategy="jeffreys")
    step = 2 if gaps else 1
    d_idx = list(range(D - step * W, D, step))
    batch = _plan(mkt, spec, d_idx, need_hf=False)
    got, work, launches = _work_delta(engine, lambda: engine.moments(batch, outputs=JEFF_OUTS, jeffreys=True))
    assert (work["add_blocks"] > 0) == (grid != "none"), work
    want = {g: _daily_grid_work(batch, *bf) for g, bf in GRIDS.items()}
    assert (work["k_rows"], work["precompute_rows"]) == want[grid], (work, want)
    assert sum(w == want[grid] for w in want.values()) == 1        # the counters tell the grids apart
    route = f"daily grid W={W} K={K}{' gaps' if gaps else ''}"
    check_windows(route, engine, mkt, batch, got, range(W), conjugate=False, jeffreys=True)
    rev = dataclasses.replace(batch, day_row=batch.day_row[::-1].copy(), span_days=batch.span_days[::-1].copy())
    back, rwork, rlaunches = _work_delta(engine, lambda: engine.moments(rev, outputs=JEFF_OUTS, jeffreys=True))
    assert rwork == work
    assert launches - rlaunches == (1 if W >= 32 else 0)          # the banded prep pass (batch_plan.cu band_ok)
    check_windows(route + " reversed", engine, mkt, rev, back, range(W), conjugate=False, jeffreys=True)


# ------------------------------------------------------------------------------------------------- intraday routes
def _days(batch, bars):
    return (batch.hf_hi - batch.hf_lo + bars - 1) // bars


def test_intraday_block_grid(engine):
    """Days of 2 bars (shorter than 8): the 64/16 row grid instead of day blocks."""
    N, W = 40, 32
    mkt = _market(N, 300, seed=501, bars=2)
    engine.upload_market(**mkt.arrays())
    spec = _spec(N, 60)
    batch = _plan(mkt, spec, list(range(300 - W, 300)), look=200)
    got, work, _ = _work_delta(engine, lambda: engine.moments(batch, outputs=CONJ_OUTS))
    assert work["add_blocks"] > 0          # K = 59 < 128: every added tile is an intraday block
    check_windows("intraday grid 64/16", engine, mkt, batch, got, range(W), spec=spec)


def test_day_blocks_with_gathered_overnight_rows(engine):
    """7-day look-back: one stored tile per trading day (no overnight return inside) + the gathered overnight rows."""
    N, W = 40, 40
    mkt = _market(N, 100, seed=502)
    engine.upload_market(**mkt.arrays())
    spec = _spec(N, 60)
    batch = _plan(mkt, spec, list(range(100 - W, 100)), look=7)
    got, work, _ = _work_delta(engine, lambda: engine.moments(batch, outputs=CONJ_OUTS))
    assert 3 <= work["add_blocks"] / W <= 6, work
    check_windows("day blocks + overnight", engine, mkt, batch, got, range(W), spec=spec)


# 64 consecutive dates from row 63: with 31 calendar days the runs have 20..22 blocks and chunks of 19, and three runs
# start late enough in a chunk to reach a third one.  With 366 days (chunks of ~253 blocks) two runs of 20 dates, 242
# rows apart, give runs of the second group that start at a chunk's last blocks.
PRESUM_DATES = {31: list(range(63, 127)), 366: list(range(300, 320)) + list(range(542, 562))}


@pytest.mark.parametrize("look,N", [(31, 40), (31, 200), (366, 24), (366, 500)])
def test_presummed_day_blocks(engine, look, N):
    """Every window adds one scanned tile per chunk its run touches -- the device's tile count is the planner's, window
    for window -- and some runs span three chunks (suffix' + the whole middle chunk + prefix).  The same batch with
    presum off (one tile per day) holds the same bound.  N = 500 with ~20k rows per window: every row against the
    tile-edge and random columns, for the three-chunk windows and both ends."""
    d_idx = PRESUM_DATES[look]
    mkt = _market(N, d_idx[-1] + 1, seed=503 + look)
    engine.upload_market(**mkt.arrays())
    spec = _spec(N, 60)
    batch = _plan(mkt, spec, d_idx, look=look)
    W = batch.n_windows
    chunks = _presum_chunks(batch)
    three = np.nonzero(chunks == 3)[0]
    assert three.size > 0
    got, work, _ = _work_delta(engine, lambda: engine.moments(batch, outputs=CONJ_OUTS))
    assert work["add_blocks"] == chunks.sum(), (work, chunks.sum())          # K = 59 < 128: no daily blocks
    windows = range(W) if N < 500 else sorted({0, W - 1, *three.tolist()})
    check_windows(f"presum {look}d N={N}", engine, mkt, batch, got, windows, spec=spec)
    days = _days(batch, 78)
    with knobs(engine, presum=0):
        plain, pw, _ = _work_delta(engine, lambda: engine.moments(batch, outputs=CONJ_OUTS))
    assert pw["add_blocks"] / W >= days.min() - 3, pw     # one tile per inner day (not the two edge days)
    windows = range(W) if N < 500 else (0, int(three[0]), W - 1)
    check_windows(f"presum off {look}d N={N}", engine, mkt, batch, plain, windows, spec=spec)


@pytest.mark.parametrize("look", [7, 31])
def test_irregular_calendar_with_missing_bars(engine, look):
    """Half days, bars absent from the calendar and NaN bars that dropna removes with the returns on both sides."""
    N, W, bars = 24, 40, 26
    mkt = _market(N, 140, seed=504 + look, bars=bars, irregular=True)
    spec = _spec(N, 60, strategy="conjugate_hf_epu_vw")
    batch = _plan(mkt, spec, list(range(140 - W, 140)), look=look)
    mkt = _with_holes(mkt, batch, np.random.default_rng(look))
    engine.upload_market(**mkt.arrays())
    got, work, _ = _work_delta(engine, lambda: engine.moments(batch, outputs=CONJ_OUTS))
    assert work["add_blocks"] > 0
    assert np.any(got["scalars"][:, SC["m"]] < batch.hf_hi - batch.hf_lo - 1)
    check_windows(f"irregular + NaN {look}d", engine, mkt, batch, got, range(W), spec=spec)


# ------------------------------------------------------------------------------------------------- workspace
def test_chunked_batch_is_bit_identical(engine):
    """A limit of two windows' workspace: the batch runs in three chunks on the same plan, bit for bit the unchunked
    result (each window's Gram job depends only on its own descriptor)."""
    N, W = 129, 6
    mkt = _market(N, 75, seed=601)
    engine.upload_market(**mkt.arrays())
    spec = _spec(N, 60)
    batch = _plan(mkt, spec, list(range(69, 75)))
    engine.set_stage_timing(True)
    try:
        engine.stage_times()
        with knobs(engine, reuse=NO_REUSE):
            one, w1, _ = _work_delta(engine, lambda: engine.moments(batch, outputs=CONJ_OUTS))
        g1 = engine.stage_times()["gram"]["launches"]
        with knobs(engine, reuse=NO_REUSE, limit=2 * _per_window(N, 78) + 64):
            three, w3, _ = _work_delta(engine, lambda: engine.moments(batch, outputs=CONJ_OUTS))
        g3 = engine.stage_times()["gram"]["launches"]
    finally:
        engine.set_stage_timing(False)
    assert w1 == w3
    assert g1 == 3 and g3 == 3 * g1                  # T, S0 and S1 launches, once per chunk: three chunks
    for k in CONJ_OUTS:
        assert np.array_equal(one[k], three[k]), k
    check_windows("chunked", engine, mkt, batch, three, range(W), spec=spec)


def test_limit_gives_up_daily_reuse(engine):
    """A store larger than half the limit: the daily phase contracts every window from scratch (batch_plan.cu:295)."""
    N, W = 64, 32
    mkt = _market(N, 300, seed=602, bars=2)
    engine.upload_market(**mkt.arrays())
    spec = _spec(N, 252, strategy="jeffreys")
    batch = _plan(mkt, spec, list(range(300 - W, 300)), need_hf=False)
    _, full, _ = _work_delta(engine, lambda: engine.moments(batch, outputs=JEFF_OUTS, jeffreys=True))
    assert full["add_blocks"] > 0
    with knobs(engine, limit=200 << 10):
        got, work, _ = _work_delta(engine, lambda: engine.moments(batch, outputs=JEFF_OUTS, jeffreys=True))
    assert work["add_blocks"] == 0, work
    check_windows("limit: no daily reuse", engine, mkt, batch, got, range(W), conjugate=False, jeffreys=True)


def test_limit_turns_presum_off(engine):
    """3 nb tiles > limit >= 2 nb tiles: the day blocks stay (one tile per day), their scans do not
    (batch_plan.cu:267)."""
    N, W = 40, 48
    mkt = _market(N, 110, seed=603)
    engine.upload_market(**mkt.arrays())
    spec = _spec(N, 60)
    batch = _plan(mkt, spec, list(range(110 - W, 110)), look=31)
    days = _days(batch, 78)
    _, pre, _ = _work_delta(engine, lambda: engine.moments(batch, outputs=CONJ_OUTS))
    assert pre["add_blocks"] / W <= 3
    with knobs(engine, limit=20 << 20):
        got, work, _ = _work_delta(engine, lambda: engine.moments(batch, outputs=CONJ_OUTS))
    assert work["add_blocks"] / W >= days.min() - 2, work
    check_windows("limit: presum off", engine, mkt, batch, got, range(W), spec=spec)


# ------------------------------------------------------------------------------------------------- pipelined
def test_pipelined_s1_matches_blocking_bits(engine):
    """The conjugate solve behind a segmented asynchronous upload (prep + Gram per segment) gives the blocking call's
    S1 and weights bit for bit, and S1 holds the bound.  The windows of the full waves solved between segments are
    factorised in place, so their S1 must leave before that solve, not after the last segment: into host memory (through
    the staging buffer) and into device memory (straight into the output) alike."""
    import torch
    N, W, segs = 40, 140, 4
    mkt = _market(N, 200, seed=701)
    spec = _spec(N, 60)
    batch = _plan(mkt, spec, list(range(60, 200)), look=7)
    outs = ("S1", "t", "rhs", "weights", "scalars", "status")
    engine.upload_market(**mkt.arrays())
    ref = engine.conjugate(batch, outputs=outs)
    pinned = {k: torch.from_numpy(np.ascontiguousarray(v)).pin_memory() for k, v in mkt.arrays().items()}
    try:
        engine.set_upload_pipeline(segs, 0)
        engine.set_stage_timing(True)
        engine.stage_times()
        engine.upload_market(**{k: v.numpy() for k, v in pinned.items()}, async_copy=True)
        got = engine.conjugate(batch, outputs=outs)
        engine.synchronize()
        gram_launches = engine.stage_times()["gram"]["launches"]
        engine.upload_market(**{k: v.numpy() for k, v in pinned.items()}, async_copy=True)
        dev = engine.conjugate(batch, outputs=outs, device_out=True)
        engine.synchronize()
        dev = {k: v.cpu().numpy() for k, v in dev.items()}
    finally:
        engine.set_stage_timing(False)
        engine.set_upload_pipeline()
    assert gram_launches > 2 * 2               # a window Gram launch per segment besides the block precomputes
    assert not got["status"].any()
    for k in outs:
        assert np.array_equal(got[k], ref[k]), k
        assert np.array_equal(dev[k], ref[k]), k
    check_windows("pipelined", engine, mkt, batch, got, range(W), spec=spec)


# ------------------------------------------------------------------------------------------------- weekly, Jorion
def test_weekly_windows(engine):
    from incorporating_different_sources_b200.windows import plan_weekly_windows
    N, W, D = 20, 30, 460
    mkt = _market(N, D, seed=801)
    spec = _spec(N, 60, freq="weekly", strategy="conjugate_hf_epu_vw")
    d_idx = list(range(D - W, D))
    rows, batch = plan_weekly_windows(spec, mkt.dates, d_idx, mkt.dates, mkt.rf, mkt.mcm, mkt.hf_ts)
    engine.upload_market(**mkt.arrays())
    engine.set_resampled(rows)
    got, work, _ = _work_delta(engine, lambda: engine.moments(batch, outputs=CONJ_OUTS))
    assert work["add_blocks"] == 0
    # the weekly rows are built on the device from the daily prices; the reference takes the oracle's rows (the same
    # correctly rounded ratios, and (1 + rf)^(7/365) - 1 for a, whose absolute rounding is far below the bound's terms)
    a_max = (1.0 + float(mkt.rf.max())) ** (7.0 / 365.0) - 1.0
    wk = {}
    for i, d in enumerate(d_idx):
        _, _, X = bo.daily_statistics(spec, mkt, d, np.arange(N))
        wk[i] = (X, np.full(X.shape[0], a_max))
    check_windows("weekly", engine, mkt, batch, got, range(W), weekly_rows=wk)


def test_jorion_centred_gram(engine):
    """Jorion's S1 is the centred Gram C = T - t t'/(n - 1) (beta = 1/m with m = n - 1 returns)."""
    N, W = 40, 32
    mkt = _market(N, 110, seed=802)
    engine.upload_market(**mkt.arrays())
    spec = _spec(N, 60, strategy="jorion")
    batch = _plan(mkt, spec, list(range(110 - W, 110)), need_hf=False)
    got = engine.jorion(batch, outputs=("S1", "t", "status"))
    assert not got["status"].any()
    check_windows("jorion C", engine, mkt, batch, got, range(W), conjugate=False, jorion=True)


# ------------------------------------------------------------------------------------------------- handle state
def test_fewer_blocks_after_more(engine):
    """Stores grow only: a batch with fewer day blocks after one with more reads none of the old tiles."""
    N = 40
    mkt = _market(N, 124, seed=901)
    engine.upload_market(**mkt.arrays())
    spec = _spec(N, 60)
    big = _plan(mkt, spec, list(range(60, 124)), look=31)
    engine.moments(big, outputs=CONJ_OUTS)
    small = _plan(mkt, spec, list(range(80, 113)), look=7)
    got, work, _ = _work_delta(engine, lambda: engine.moments(small, outputs=CONJ_OUTS))
    assert 0 < work["add_blocks"] / small.n_windows <= 6
    check_windows("fewer blocks after more", engine, mkt, small, got, range(small.n_windows), spec=spec)


def test_smaller_market_after_larger(engine):
    """ld, hf_extra_rows and the intraday capacity shrink in use: N = 257 with 120 days, then N = 33 with 95 days."""
    big = _market(257, 120, seed=902)
    engine.upload_market(**big.arrays())
    spec = _spec(257, 60)
    engine.moments(_plan(big, spec, list(range(120 - 48, 120)), look=31), outputs=CONJ_OUTS)
    mkt = _market(33, 95, seed=903)
    engine.upload_market(**mkt.arrays())
    spec = _spec(33, 60)
    for look in (7, 31):
        batch = _plan(mkt, spec, list(range(95 - 32, 95)), look=look)
        got, work, _ = _work_delta(engine, lambda: engine.moments(batch, outputs=CONJ_OUTS))
        assert work["add_blocks"] > 0
        check_windows(f"small after large {look}d", engine, mkt, batch, got, range(32), spec=spec)


def test_pool_with_permuted_columns(engine):
    N_pool, N, W = 64, 40, 40
    pool = _market(N_pool, 100, seed=904)
    cols = np.random.default_rng(5).permutation(N_pool)[:N]
    mkt = pool.columns(cols)
    spec = _spec(N, 60)
    batch = _plan(mkt, spec, list(range(100 - W, 100)), look=7)
    engine.upload_pool(prices=pool.prices, rf_row=pool.rf_row, caps=pool.caps, hf_prices=pool.hf_prices)
    try:
        engine.select_market(cols, 0, pool.prices.shape[0], 0, pool.hf_prices.shape[0])
        got = engine.moments(dataclasses.replace(batch, prior_n=np.full(W, 150.0)), outputs=CONJ_OUTS)
        assert np.all(got["scalars"][:, SC["n0"]] == 150.0)
        check_windows("pool + select", engine, mkt, batch, got, range(W))
    finally:
        engine.upload_pool(None, None)
