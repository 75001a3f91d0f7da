"""The Jeffreys / Jorion chain (jeffreys_chain.cu) on its own: windows of consecutive dates solved relative to a
factorised base window, held window by window to the extended-precision reference and a-priori bound of
tests/_chain_ref.py.  Panel and cp.async-ring edges up to N = 640 (the largest N whose right-hand-side block fits
shared memory), every group size with the smallest batch that chains, the planner's rank guard exactly at its margin,
an ill-conditioned but regular window, Jorion's scalars, determinism, and the status of windows whose base failed or
whose own matrix is singular.  Every case asserts from the library's work counters which route it took."""
import numpy as np
import pytest

from tests import _chain_ref as cr
from tests import _solver_ref as sr

pytestmark = pytest.mark.gpu

U = cr.U
OUTS = ("weights", "nu", "w1", "scalars", "status")
GAMMA = 3.0
WORST = {}                 # case -> output -> worst |E| / bound seen (printed at the end of the module)


@pytest.fixture(scope="module")
def engine():
    from incorporating_different_sources_b200.engine import BayesEngine
    sr.require_extended_precision()
    eng = BayesEngine(0)
    yield eng
    eng.close()
    if WORST:
        print("\nworst |E| / bound per case:")
        for case, d in WORST.items():
            print(f"  {case:34s} " + " ".join(f"{k}={v:.3g}" for k, v in sorted(d.items())))


def margin(N, G):
    """The smallest rolling window the planner chains with group G: n - 1 = N + 2G + 8."""
    return N + 2 * G + 9


def _assert_ratio(case, name, r, w):
    d = WORST.setdefault(case, {})
    d[name] = max(d.get(name, 0.0), r)
    assert r < 1.0, f"{case}: {name} of window {w} is {r:.3g} x its bound"


def run(engine, mkt, d_idx, n, G, jorion=False, chained=True):
    """One batched call with chain group G; asserts the route from the work counters."""
    from incorporating_different_sources_b200.engine import upload_synthetic
    N, W = mkt.prices.shape[1], len(d_idx)
    upload_synthetic(engine, mkt)
    batch = cr.plan(mkt, cr.jeffreys_spec(N, n, "jorion" if jorion else "jeffreys"), d_idx)
    try:
        engine.set_jeffreys_chain(G)
        engine.solve_work()
        got = (engine.jorion if jorion else engine.jeffreys)(batch, outputs=OUTS)
        work = engine.solve_work()
    finally:
        engine.set_jeffreys_chain(8)
    n_base = -(-W // G) if chained else W
    assert work == {"factored": float(n_base), "chained": float(W - n_base)}, work
    return got, batch


def groups_to_check(W, G, N):
    """Every group, or at N >= 500 the first, a middle and the last one (the longdouble reference is the cost)."""
    starts = list(range(0, W, G))
    if N >= 500:
        starts = sorted({starts[0], starts[len(starts) // 2], starts[-1]})
    return starts


def check(case, mkt, batch, got, G, jorion=False, starts=None, skip=(), chained=True):
    """Hold every window of the listed groups to the chain's bound (the solver's bound for base windows and on the
    per-window path).  Windows in ``skip`` are not checked."""
    from incorporating_different_sources_b200._lib import SCAL, SCAL_JORION
    N, W, n = mkt.prices.shape[1], batch.n_windows, int(batch.rolling_window)
    refs = cr.WindowRefs(cr.log_returns(mkt.prices), cr.rf_rows(mkt), batch, jorion=jorion)
    starts = groups_to_check(W, G, N) if starts is None else starts
    for b in starts:
        Jb, tb = refs(b)
        kb, eb = cr.kappa2(Jb.value), cr.eta(Jb)
        for w in range(b, min(b + G, W)):
            J, t = (Jb, tb) if w == b else refs(w)
            if w in skip:
                continue
            k = w - b
            kw = cr.kappa2(J.value) if k else kb
            eta_in = max(eb, cr.eta(J)) + cr.eta(t)
            eps = cr.chain_bound(N, k, kb, kw, eta_in) if k and chained else cr.solver_bound(N, kw, eta_in)
            if not jorion:
                x_ref = cr.refined_solve(J.value, t.value)
                for key in ("w1", "nu"):
                    _assert_ratio(case, key, sr.forward_error(got[key][w], x_ref) / eps, w)
                _assert_ratio(case, "weights", sr.forward_error(got["weights"][w], x_ref / cr.LD(GAMMA)) / (eps + 2 * U), w)
                v1 = np.asarray(x_ref, dtype=cr.LD) @ t.value
                err = abs(float(cr.LD(got["scalars"][w][SCAL["v1"]]) - v1))
                _assert_ratio(case, "v1", err / cr.v1_bound(x_ref, eps, t), w)
            else:
                r = sr.jorion_reference(J.value, t.value, n - 1, GAMMA, kw, eps=eps)
                _assert_ratio(case, "w1", sr.forward_error(got["w1"][w], r["y"].v) / eps, w)
                for key in ("weights", "nu"):
                    e = np.abs(got[key][w].astype(cr.LD) - r[key].v) / (2 * r[key].e)
                    _assert_ratio(case, key, float(np.max(e)), w)
                for name, slot in SCAL_JORION.items():
                    e = abs(cr.LD(got["scalars"][w][slot]) - r[name].v) / (2 * r[name].e)
                    _assert_ratio(case, name, float(e), w)


# ------------------------------------------------------------------------------------------- 1. panel and ring edges
EDGES = [  # (N, n, W): G = 8; n at the margin or 1008; W mod 8 in {0, 1, 7}
    (1, margin(1, 8), 16), (2, 1008, 17), (31, margin(31, 8), 23), (32, 1008, 16), (33, margin(33, 8), 17),
    (63, margin(63, 8), 23), (64, 1008, 24), (65, margin(65, 8), 17), (200, margin(200, 8), 23), (500, 1008, 24),
    (639, margin(639, 8), 17), (640, margin(640, 8), 23), (640, 1008, 16)]


@pytest.mark.parametrize("N,n,W", EDGES)
def test_panel_edges(engine, N, n, W):
    mkt, d_idx = cr.chain_market(N, n, W, seed=4000 + N + n)
    got, batch = run(engine, mkt, d_idx, n, 8)
    assert not got["status"].any()
    check(f"edge N={N} n={n} W={W}", mkt, batch, got, 8)


def test_shared_memory_limit(engine):
    """N = 641 qualifies in every other respect, but its right-hand-side block does not fit: every window is factorised."""
    N, n, W = 641, 1008, 16
    mkt, d_idx = cr.chain_market(N, n, W, seed=641)
    got, batch = run(engine, mkt, d_idx, n, 8, chained=False)
    assert not got["status"].any()
    check("smem N=641", mkt, batch, got, 8, starts=[0], chained=False)


# ------------------------------------------------------------------------------------------- 2. group sizes
@pytest.mark.parametrize("N", [33, 96])
@pytest.mark.parametrize("G", [2, 3, 4, 5, 6, 7, 8])
def test_group_sizes(engine, N, G):
    """W = 2G chains, W = 2G - 1 factorises every window, W = 3G - 1 ends with a partial group of G - 1 windows."""
    n = 252
    mkt, d_idx = cr.chain_market(N, n, 3 * G - 1, seed=5000 + 10 * N + G)
    for W, chained in ((2 * G, True), (2 * G - 1, False), (3 * G - 1, True)):
        got, batch = run(engine, mkt, d_idx[:W], n, G, chained=chained)
        assert not got["status"].any()
        check(f"group N={N} G={G}", mkt, batch, got, G, chained=chained)


# ------------------------------------------------------------------------------------------- 3. rank guard
@pytest.mark.parametrize("G", [2, 5, 8])
def test_rank_guard(engine, G):
    """n - 1 = N + 2G + 8 chains and every chained window meets the bound; one row less factorises every window."""
    N = 40
    W = 2 * G + 3
    for n, chained in ((margin(N, G), True), (margin(N, G) - 1, False)):
        mkt, d_idx = cr.chain_market(N, n, W, seed=6000 + G + n)
        got, batch = run(engine, mkt, d_idx, n, G, chained=chained)
        assert not got["status"].any()
        check(f"guard G={G} {'chain' if chained else 'plain'}", mkt, batch, got, G, chained=chained)


def test_flat_asset_at_positive_rate(engine):
    """An asset flat over a whole window while rf > 0: its excess return is -a, the window is regular but
    ill-conditioned (cond(J) ~ 1e7); status 0 and within the bound, the neighbours (one row of the asset moving) too."""
    N, n, G, W = 40, 120, 8, 16
    mkt, d_idx = cr.chain_market(N, n, W, seed=31)
    day = d_idx[11]
    cr.flatten(mkt, 5, day - n + 2, day + 1)
    got, batch = run(engine, mkt, d_idx, n, G)
    assert not got["status"].any()
    J, _ = cr.WindowRefs(cr.log_returns(mkt.prices), cr.rf_rows(mkt), batch)(11)
    assert cr.kappa2(J.value) > 1e6
    check("flat asset, rf > 0", mkt, batch, got, G)


# ------------------------------------------------------------------------------------------- 4. Jorion
@pytest.mark.parametrize("N", [33, 200, 640])
@pytest.mark.parametrize("G", [3, 8])
@pytest.mark.parametrize("at_margin", [True, False])
def test_jorion(engine, N, G, at_margin):
    """y = C^-1 t (w1), nu, weights and the Bayes-Stein scalars of every checked window against jorion_reference
    carrying the chain's bound."""
    n = margin(N, G) if at_margin else 1008
    W = 2 * G + 2
    mkt, d_idx = cr.chain_market(N, n, W, seed=7000 + N + G + n)
    got, batch = run(engine, mkt, d_idx, n, G, jorion=True)
    assert not got["status"].any()
    check(f"jorion N={N} G={G} n={n}", mkt, batch, got, G, jorion=True)


# ------------------------------------------------------------------------------------------- 5. outputs, determinism
def test_base_windows_with_and_without_chain(engine):
    """The base windows are factorised either way: with the chain on and off they meet the solver's bound."""
    N, n, W, G = 65, 300, 24, 8
    mkt, d_idx = cr.chain_market(N, n, W, seed=65)
    on, batch = run(engine, mkt, d_idx, n, G)
    off, _ = run(engine, mkt, d_idx, n, 0, chained=False)
    assert not on["status"].any() and not off["status"].any()
    check("bases, chain on", mkt, batch, on, G, starts=[0, 8, 16], skip=set(range(W)) - {0, 8, 16})
    check("bases, chain off", mkt, batch, off, G, starts=[0, 8, 16], skip=set(range(W)) - {0, 8, 16}, chained=False)


@pytest.mark.parametrize("jorion", [False, True])
def test_deterministic(engine, jorion):
    """No atomics and a fixed reduction order: the same chained batch twice gives the same bits."""
    N, n, W, G = 200, 400, 24, 8
    mkt, d_idx = cr.chain_market(N, n, W, seed=200)
    a, _ = run(engine, mkt, d_idx, n, G, jorion=jorion)
    b, _ = run(engine, mkt, d_idx, n, G, jorion=jorion)
    for k in OUTS:
        assert np.array_equal(a[k], b[k]), k


# ------------------------------------------------------------------------------------------- 6. status
N_ST, n_ST, G_ST, W_ST, B_ST, ASSET = 40, 120, 8, 24, 8, 7


@pytest.mark.parametrize("jorion", [False, True])
def test_status_failed_base(engine, jorion):
    """rf = 0 and an asset flat exactly over the return rows of group 1's base window (moving again from day_b + 1):
    the base reports ASSET + 1 and so do its chained windows; the other groups report 0 and meet the bound.  The
    per-window path reports ASSET + 1 for the base only."""
    mkt, d_idx = cr.chain_market(N_ST, n_ST, W_ST, seed=88, rf_zero=True)
    day_b = d_idx[B_ST]
    cr.flatten(mkt, ASSET, day_b - n_ST + 2, day_b + 1)
    got, batch = run(engine, mkt, d_idx, n_ST, G_ST, jorion=jorion)
    bad = set(range(B_ST, B_ST + G_ST))
    for w in range(W_ST):
        assert got["status"][w] == (ASSET + 1 if w in bad else 0), (w, got["status"][w])
    check(f"failed base, jorion={jorion}", mkt, batch, got, G_ST, jorion=jorion, starts=[0, 16])
    plain, _ = run(engine, mkt, d_idx, n_ST, 0, jorion=jorion, chained=False)
    for w in range(W_ST):
        assert plain["status"][w] == (ASSET + 1 if w == B_ST else 0), (w, plain["status"][w])


@pytest.mark.parametrize("jorion", [False, True])
def test_status_singular_chained_windows(engine, jorion):
    """rf = 0 and an asset flat on return rows [day_b - n + 5, day_b + 6) of group 1: windows b+3 .. b+5 are exactly
    singular and report N + 1 (singular relative to the base); b+1, b+2, b+6 and b+7 report 0 and meet the bound.  The
    per-window path reports ASSET + 1 for the singular windows."""
    mkt, d_idx = cr.chain_market(N_ST, n_ST, W_ST, seed=89, rf_zero=True)
    day_b = d_idx[B_ST]
    cr.flatten(mkt, ASSET, day_b - n_ST + 5, day_b + 6)
    sing = {B_ST + 3, B_ST + 4, B_ST + 5}
    got, batch = run(engine, mkt, d_idx, n_ST, G_ST, jorion=jorion)
    for w in range(W_ST):
        assert got["status"][w] == (N_ST + 1 if w in sing else 0), (w, got["status"][w])
    check(f"singular chained, jorion={jorion}", mkt, batch, got, G_ST, jorion=jorion, skip=sing)
    plain, _ = run(engine, mkt, d_idx, n_ST, 0, jorion=jorion, chained=False)
    for w in range(W_ST):
        assert plain["status"][w] == (ASSET + 1 if w in sing else 0), (w, plain["status"][w])
