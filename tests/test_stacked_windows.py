"""Host planning of stacked working markets (windows of different asset sets in one batch): ``stack_windows`` relocates
the per-set plan into one block per window, and ``stack_batches`` keeps each batch to one N and a byte budget."""
import numpy as np
import pytest

from incorporating_different_sources_b200.synthetic import generate_market
from incorporating_different_sources_b200.windows import (HF_LOOKBACK_DAYS, plan_daily_windows, plan_weekly_windows,
                                                          stack_batches, stack_windows)

_DAY = np.timedelta64(1, "D")


def _spec(strategy, n, freq):
    return {"weighting_strategy": strategy, "rolling_window": n, "rolling_window_frequency": freq,
            "mcm_scaling": 1.0, "risk_aversion": 2.0}


def _sets(rng, n_pool, size, dates_pos):
    """Random top-k universes: every rebalance date gets one of a few column sets, some sets repeat."""
    pool = [tuple(sorted(rng.choice(n_pool, size, replace=False))) for _ in range(6)]
    groups = {}
    for d in dates_pos:
        groups.setdefault(pool[int(rng.integers(len(pool)))], []).append(int(d))
    return list(groups.items())


def _per_set_daily(spec, mkt, d_idx, look, need_hf):
    """The plan of one set as backtest._batched_weights makes it for its own select_market slice; the slice and the
    shifted batch are also checked against the set's trade dates and look-back, searched directly."""
    from incorporating_different_sources_b200 import backtest as bt
    n = spec["rolling_window"]
    _, b = bt._plan_windows(spec, spec["weighting_strategy"], mkt.dates, np.asarray(d_idx), mkt.hf_ts, mkt.dates, mkt.rf,
                            look)
    day_lo, day_hi, hf_lo, hf_hi = bt._set_slice(b, mkt.n_days, len(mkt.hf_ts))
    assert (day_lo, day_hi) == (min(d_idx) - (n - 1), max(d_idx) + 1)
    want_lo = want_hi = 0
    if need_hf:
        D = look if look is not None else HF_LOOKBACK_DAYS[spec["rolling_window_frequency"]]
        want_lo = max(int(np.searchsorted(mkt.hf_ts, mkt.dates[min(d_idx)] - D * _DAY + _DAY, side="right")) - 1, 0)
        want_hi = int(np.searchsorted(mkt.hf_ts, mkt.dates[max(d_idx)] + _DAY, side="right"))
    assert (hf_lo, hf_hi) == (want_lo, want_hi)
    ref = plan_daily_windows(spec, mkt.dates, d_idx, mkt.hf_ts if need_hf else None, hf_lookback_days=look,
                             need_hf=need_hf, row_offset=day_lo, hf_row_offset=hf_lo)
    for name in ("day_row", "span_days", "hf_lo", "hf_hi"):
        a, r = getattr(b, name), getattr(ref, name)
        assert (a is None and r is None) or (a.dtype == r.dtype and np.array_equal(a, r)), name
    return b, day_lo, hf_lo


def _check_tiling(stk):
    dl = stk.day_hi - stk.day_lo
    assert stk.day_off[0] == 0 and np.all(dl > 0)
    assert np.array_equal(stk.day_off[1:], stk.day_off[:-1] + dl[:-1])
    if stk.hf_lo is not None:
        hl = stk.hf_hi - stk.hf_lo
        assert stk.hf_off[0] == 0 and np.all(hl > 0)
        assert np.array_equal(stk.hf_off[1:], stk.hf_off[:-1] + hl[:-1])


def _in_block(stk, w, rows_lo, rows_hi, hf=False):
    off, lo, hi = (stk.hf_off, stk.hf_lo, stk.hf_hi) if hf else (stk.day_off, stk.day_lo, stk.day_hi)
    assert off[w] <= rows_lo and rows_hi <= off[w] + hi[w] - lo[w]


@pytest.mark.parametrize("strategy,look", [("conjugate_hf_vix_vw", 7), ("conjugate_hf_epu_ew", None), ("jeffreys", None)])
@pytest.mark.parametrize("seed", [1, 2])
def test_daily_windows_relocate_to_their_blocks(strategy, look, seed):
    rng = np.random.default_rng(seed)
    mkt = generate_market(20, 160, seed=seed)
    n = 40
    spec = _spec(strategy, n, "daily")
    need_hf = strategy.startswith("conjugate")
    sets = _sets(rng, 20, 7, rng.choice(np.arange(n + 10, 160), 30, replace=False))
    d_all = [d for _, ds in sets for d in ds]
    plan = plan_daily_windows(spec, mkt.dates, d_all, mkt.hf_ts if need_hf else None, hf_lookback_days=look, need_hf=need_hf)
    stk = stack_windows(plan)
    _check_tiling(stk)
    assert stk.resampled is None and (stk.hf_lo is None) == (not need_hf)
    b = stk.batch
    w = 0
    for _, ds in sets:
        ref, day_lo, hf_lo = _per_set_daily(spec, mkt, ds, look, need_hf)
        for j in range(len(ds)):
            assert b.day_row[w] - stk.day_off[w] + stk.day_lo[w] == ref.day_row[j] + day_lo
            assert b.span_days[w] == ref.span_days[j]
            _in_block(stk, w, b.day_row[w] - (n - 1), b.day_row[w] + 1)
            if need_hf:
                assert b.hf_lo[w] - stk.hf_off[w] + stk.hf_lo[w] == ref.hf_lo[j] + hf_lo
                assert b.hf_hi[w] - stk.hf_off[w] + stk.hf_lo[w] == ref.hf_hi[j] + hf_lo
                assert b.hf_lo[w] - stk.hf_off[w] in (0, 1)          # the one row in front of the first bar
                _in_block(stk, w, b.hf_lo[w], b.hf_hi[w], hf=True)
            w += 1
    assert w == b.n_windows
    for name in ("rolling_window", "mcm_index", "mcm_scaling", "risk_aversion", "prior_weights", "resampled"):
        assert getattr(b, name) == getattr(plan, name)


@pytest.mark.parametrize("strategy", ["conjugate_hf_vix_vw", "jeffreys"])
@pytest.mark.parametrize("seed", [3, 4])
def test_weekly_windows_relocate_with_their_resampled_rows(strategy, seed):
    rng = np.random.default_rng(seed)
    mkt = generate_market(16, 300, seed=seed)
    n = 20
    spec = _spec(strategy, n, "weekly")
    need_hf = strategy.startswith("conjugate")
    sets = _sets(rng, 16, 6, rng.choice(np.arange(130, 300), 25, replace=False))
    d_all = [d for _, ds in sets for d in ds]
    kw = dict(hf_lookback_days=7) if need_hf else dict(need_hf=False)
    rows, plan = plan_weekly_windows(spec, mkt.dates, d_all, mkt.dates, mkt.rf, None, mkt.hf_ts if need_hf else None, **kw)
    stk = stack_windows(plan, rows)
    _check_tiling(stk)
    rs, b = stk.resampled, stk.batch
    D = int((stk.day_hi - stk.day_lo).sum())
    assert rs.num_row.min() >= 0 and rs.num_row.max() < D and rs.den_row.max() < D
    w = 0
    for _, ds in sets:
        # the per-set plan: the whole calendar and its own ResampledRows (bp_set_resampled on the set's market)
        ref_rows, ref = plan_weekly_windows(spec, mkt.dates, ds, mkt.dates, mkt.rf, None, mkt.hf_ts if need_hf else None, **kw)
        for j in range(len(ds)):
            shift = stk.day_lo[w] - stk.day_off[w]
            mine = np.r_[np.arange(b.day_row[w] - (n - 3), b.day_row[w] + 1), b.extra_row[w]]
            theirs = np.r_[np.arange(ref.day_row[j] - (n - 3), ref.day_row[j] + 1), ref.extra_row[j]]
            assert mine.min() >= 1                                          # row 0 is never read
            assert np.array_equal(rs.num_row[mine] + shift, ref_rows.num_row[theirs])
            assert np.array_equal(rs.den_row[mine] + shift, ref_rows.den_row[theirs])
            assert np.array_equal(rs.rf_row[mine], ref_rows.rf_row[theirs])   # the partial week's look-ahead label too
            for r in (rs.num_row[mine], rs.den_row[mine]):
                _in_block(stk, w, r.min(), r.max() + 1)
            assert b.caps_row[w] + shift == ref.caps_row[j]
            _in_block(stk, w, b.caps_row[w], b.caps_row[w] + 1)
            assert b.span_days[w] == ref.span_days[j]
            if need_hf:
                assert b.hf_lo[w] - stk.hf_off[w] + stk.hf_lo[w] == ref.hf_lo[j]
                assert b.hf_hi[w] - stk.hf_off[w] + stk.hf_lo[w] == ref.hf_hi[j]
                _in_block(stk, w, b.hf_lo[w], b.hf_hi[w], hf=True)
            w += 1
    assert w == b.n_windows
    # the windows' resampled rows do not overlap: every window reads n-1 rows of its own
    assert len(rs.num_row) == 1 + b.n_windows * (n - 1)


def test_daily_window_without_enough_history():
    mkt = generate_market(4, 60, seed=5)
    b = plan_daily_windows(_spec("jeffreys", 10, "daily"), mkt.dates, [9, 30], need_hf=False)
    b.day_row[0] = 5
    with pytest.raises(ValueError, match="needs 9 rows before"):
        stack_windows(b)


def test_batches_hold_one_n_and_respect_the_budget():
    rng = np.random.default_rng(6)
    n_cols = rng.choice([10, 50, 49, 130], 200)
    nbytes = rng.integers(1, 100, 200)
    batches = stack_batches(n_cols, nbytes, 400)
    seen = np.concatenate(batches)
    assert np.array_equal(np.sort(seen), np.arange(200))
    for pos in batches:
        assert len(set(n_cols[pos].tolist())) == 1
        assert nbytes[pos].sum() <= 400 or len(pos) == 1
        assert np.all(np.diff(pos) > 0)
    # windows of one N keep their order; a window larger than the budget is a batch of its own
    assert [len(p) for p in stack_batches([5, 5, 5], [10, 500, 10], 100)] == [1, 1, 1]
    assert [p.tolist() for p in stack_batches([5, 7, 5], [1, 1, 1], 100)] == [[0, 2], [1]]


class _StubEngine:
    """Stands in for BayesEngine in ``backtest._batched_weights``: Jeffreys "weights" of window w are
    1000 * pool column + pool row of its trade date, found through whichever working market is selected, and the
    status is non-zero on the trade-date rows listed in ``bad``."""
    condition_estimate = False

    def __init__(self, stack_max, bad=()):
        self.stack_max_windows = stack_max
        self.bad = set(bad)
        self.stacked_calls = 0

    def upload_pool(self, prices, rf_row, caps=None, hf_prices=None):
        pass

    def select_market(self, cols, day_lo, day_hi, hf_lo, hf_hi):
        self.market = ("set", np.asarray(cols), day_lo)

    def select_windows(self, cols, day_ranges, hf_ranges=None):
        days = np.asarray(day_ranges)
        off = np.r_[0, np.cumsum(days[:, 1] - days[:, 0])[:-1]]
        self.market = ("stack", np.asarray(cols), days[:, 0] - off)
        self.stacked_calls += 1

    def jeffreys(self, batch, outputs):
        kind, cols, shift = self.market
        d = batch.day_row.astype(np.int64) + shift
        cols = np.broadcast_to(cols, (batch.n_windows, cols.shape[-1]))
        return {"weights": cols * 1000.0 + d[:, None],
                "status": np.asarray([r in self.bad for r in d], dtype=np.int32)}


def _mixed_backtest():
    from incorporating_different_sources_b200.synthetic import generate_market
    mkt = generate_market(12, 120, seed=12)
    md = mkt.market_data()
    spec = {"weighting_strategy": "jeffreys", "rolling_window": 20, "rolling_window_frequency": "daily",
            "risk_aversion": 1.0}
    reb_pos = list(range(40, 100))
    t = mkt.tickers
    # a small set of 5 stocks, then a large set (its own call), then small sets of 4 and 5 stocks
    universes = [t[0:5]] * 3 + [t[5:10]] * 40 + [t[1:5]] * 4 + [t[2:7]] * 5 + [t[0:4]] * 2 + [t[7:12]] * 6
    return md, spec, reb_pos, universes


@pytest.mark.parametrize("stack_max", [15, 0])
def test_backtest_weights_with_small_sets_of_different_sizes(stack_max):
    from incorporating_different_sources_b200 import backtest as bt
    md, spec, reb_pos, universes = _mixed_backtest()
    eng = _StubEngine(stack_max)
    counts = {}
    W, member = bt._batched_weights(eng, spec, md, md["stock_prices_df"].index, reb_pos, universes, counts=counts)
    pos = {c: i for i, c in enumerate(md["stock_prices_df"].columns)}
    for r, names in enumerate(universes):
        cols = sorted(pos[n] for n in names)
        want = np.zeros(W.shape[1])
        want[cols] = np.asarray(cols) * 1000.0 + reb_pos[r]
        assert np.array_equal(W[r], want), r
        assert member[r].sum() == len(cols)
    if stack_max:
        # 20 windows of small sets with 4 and 5 stocks: one stacked call per N
        assert counts == {"stacked_windows": 20, "stacked_calls": 2} and eng.stacked_calls == 2
    else:
        assert counts == {"stacked_windows": 0, "stacked_calls": 0}


@pytest.mark.parametrize("bad_sets,first", [((3, 1), 1), ((3, 2), 2), ((0, 4), 0)])
def test_backtest_failures_raise_in_set_order(bad_sets, first):
    """Whether a set is stacked or not, the first failing set in order of first appearance is the one reported."""
    from incorporating_different_sources_b200 import backtest as bt
    md, spec, reb_pos, universes = _mixed_backtest()
    starts = [0, 3, 43, 47, 52, 54]                   # first rebalance index of each set
    dates = md["stock_prices_df"].index
    msgs = []
    for stack_max in (15, 0):
        eng = _StubEngine(stack_max, bad={reb_pos[starts[k] + 1] for k in bad_sets})
        with pytest.raises(np.linalg.LinAlgError) as e:
            bt._batched_weights(eng, spec, md, dates, reb_pos, universes)
        msgs.append(str(e.value))
    assert msgs[0] == msgs[1]
    assert str(dates[reb_pos[starts[first] + 1]].date()) in msgs[0]
