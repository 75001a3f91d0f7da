"""The reference and bound of tests/_chain_ref.py on the CPU: the longdouble reference against mpmath, and a float64
emulation of jeffreys_chain.cu's algorithm (column layout, C^-1, Gauss-Jordan with the kernel's pivoting) held to the
bound over the shapes of tests/test_gpu_chain.py.  The emulation also places the kernel's singular-pivot threshold
TAU between exactly singular windows and the worst regular ones."""
import numpy as np
import pytest
import scipy.linalg as sla

from tests import _chain_ref as cr
from tests import _gram_ref as gr

N_GRID = [  # (N, n, W, G): the panel edges at the rank guard's margin (n - 1 = N + 2G + 8) or n = 1008
    (1, 26, 16, 8), (2, 1008, 17, 8), (31, 56, 23, 8), (33, 58, 17, 8), (64, 1008, 24, 8), (65, 90, 17, 8),
    (200, 225, 23, 8), (96, 109, 6, 2), (33, 50, 14, 4)]


def _group_errors(N, n, W, G, seed, jorion=False, flat=None, rf_zero=False):
    """Emulate every group of the batch; returns [(window, k, rel_err / bound, rel_pivot)]."""
    mkt, d_idx = cr.chain_market(N, n, W, seed, rf_zero=rf_zero)
    if flat is not None:
        flat(mkt, d_idx)
    batch = cr.plan(mkt, cr.jeffreys_spec(N, n), d_idx)
    lr = cr.log_returns(mkt.prices)
    refs = cr.WindowRefs(lr, cr.rf_rows(mkt), batch, jorion=jorion)
    beta_den = float(n - 1 if jorion else n)
    out = []
    for b in range(0, W, G):
        nb = min(G, W - b) - 1
        JT = [refs(b + k) for k in range(nb + 1)]
        Jb = np.asarray(JT[0][0].value, dtype=np.float64)
        Lfac = np.linalg.cholesky(Jb)
        pv, tv = [], []
        for k in range(nb + 1):
            rows = gr.daily_return_rows(int(batch.day_row[b + k]), n)
            a = gr.daily_adjustments(cr.rf_rows(mkt), rows, int(batch.span_days[b + k]))
            L = lr[rows]
            pv.append(L.T @ a - 0.5 * (a @ a))
            tv.append((L - a[:, None]).sum(axis=0))
        res = cr.emulate_group(Lfac, lr, pv, tv, int(batch.day_row[b]), n, nb, beta_den)
        kb = cr.kappa2(JT[0][0].value)
        eb = cr.eta(JT[0][0])
        for k in range(1, nb + 1):
            J, t = JT[k]
            kw = cr.kappa2(J.value)
            r = res[k - 1]
            if not np.isfinite(kw):
                out.append((b + k, k, np.inf, r["rel_pivot"]))
                continue
            x_ref = cr.refined_solve(J.value, t.value)
            eps = cr.chain_bound(N, k, kb, kw, max(eb, cr.eta(J)) + cr.eta(t))
            err = float(np.max(np.abs(r["x"].astype(cr.LD) - x_ref)) / np.max(np.abs(x_ref)))
            out.append((b + k, k, err / eps, r["rel_pivot"]))
    return out


def test_reference_matches_mpmath():
    """J, t and J^-1 t of small windows against 40-digit arithmetic on the same log returns and adjustments."""
    mpmath = pytest.importorskip("mpmath")
    mpmath.mp.dps = 40
    N, n, W = 5, 14, 3
    mkt, d_idx = cr.chain_market(N, n, W, seed=11)
    batch = cr.plan(mkt, cr.jeffreys_spec(N, n), d_idx)
    lr = cr.log_returns(mkt.prices)
    rf = cr.rf_rows(mkt)
    for jorion in (False, True):
        refs = cr.WindowRefs(lr, rf, batch, jorion=jorion)
        den = n - 1 if jorion else n
        for i in range(W):
            J, t = refs(i)
            rows = gr.daily_return_rows(int(batch.day_row[i]), n)
            a = gr.daily_adjustments(rf, rows, int(batch.span_days[i]))
            X = [[mpmath.mpf(float(lr[r, j])) - mpmath.mpf(float(a[q])) for j in range(N)] for q, r in enumerate(rows)]
            tm = [sum(X[q][j] for q in range(len(rows))) for j in range(N)]
            Jm = mpmath.matrix(N, N)
            for p in range(N):
                for j in range(N):
                    Jm[p, j] = sum(X[q][p] * X[q][j] for q in range(len(rows))) - tm[p] * tm[j] / den
            xm = mpmath.lu_solve(Jm, mpmath.matrix(tm))
            x = cr.refined_solve(J.value, t.value)
            for p in range(N):
                assert abs(float(mpmath.mpf(str(t.value[p])) - tm[p])) <= 1e-17 * float(abs(tm[p])) + 1e-19
                for j in range(N):
                    assert abs(float(mpmath.mpf(str(J.value[p, j])) - Jm[p, j])) <= 1e-17 * float(mpmath.norm(Jm, 1))
                assert abs(float(mpmath.mpf(str(x[p])) - xm[p])) <= 1e-15 * float(mpmath.norm(xm, mpmath.inf))


def test_chain_reference_jorion_formulas():
    """jorion_reference with a longdouble C and the chain's eps: y = C^-1 t and z = C^-1 1 carry eps."""
    from tests import _solver_ref as sr
    rng = np.random.default_rng(3)
    C, t, m = sr.jorion_problem(12, rng)
    r = sr.jorion_reference(C.astype(cr.LD), t, m, 2.0, sr.kappa2(C), eps=1e-9)
    assert np.allclose(np.asarray(r["y"].v, dtype=np.float64), sla.solve(C, t), rtol=1e-10)
    assert float(np.max(r["y"].e)) == pytest.approx(1e-9 * float(np.max(np.abs(r["y"].v))))


@pytest.mark.parametrize("N,n,W,G", N_GRID)
def test_emulated_chain_within_bound(N, n, W, G):
    for jorion in (False, True):
        for w, k, ratio, rel in _group_errors(N, n, W, G, seed=900 + N, jorion=jorion):
            assert ratio < 1.0, f"jorion={jorion} window {w} (k={k}): {ratio:.3g} x the bound"
            assert rel > 1e3 * cr.TAU, f"regular window {w} would be flagged: relative pivot {rel:.3g}"


def _singular_chained(b, asset):
    def flat(mkt, d_idx):
        day_b = d_idx[b]
        n = len(mkt.dates) - len(d_idx) - 3
        cr.flatten(mkt, asset, day_b - n + 5, day_b + 6)
    return flat


@pytest.mark.parametrize("N,n,G", [(40, 120, 8), (40, 65, 8), (33, 200, 8)])
def test_threshold_separates_singular_windows(N, n, G):
    """rf = 0 and one asset flat on return rows [day_b - n + 5, day_b + 6): windows b+3 .. b+5 are exactly singular
    and their relative pivots fall below TAU / 1e3; the group's other windows stay above 1e3 TAU and within the bound."""
    W, b, asset = 2 * G, G, 7
    for jorion in (False, True):
        res = _group_errors(N, n, W, G, seed=77, jorion=jorion, flat=_singular_chained(b, asset), rf_zero=True)
        for w, k, ratio, rel in res:
            if w in (b + 3, b + 4, b + 5):
                assert rel < 1e-3 * cr.TAU, (w, rel)
            else:
                assert ratio < 1.0 and rel > 1e3 * cr.TAU, (w, ratio, rel)


def test_threshold_keeps_flat_asset_at_positive_rate():
    """An asset flat over a whole window while rf > 0 (its excess return is -a, cond(J) ~ 1e7): regular, unflagged,
    within the bound."""
    N, n, G, W = 40, 120, 8, 16

    def flat(mkt, d_idx):
        day = d_idx[11]
        cr.flatten(mkt, 5, day - n + 2, day + 1)
    res = _group_errors(N, n, W, G, seed=31, flat=flat)
    assert min(r[3] for r in res) > 1e3 * cr.TAU
    assert max(r[2] for r in res) < 1.0
