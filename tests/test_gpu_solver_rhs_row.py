"""Where the right-hand side rides along through the Cholesky factorisation (chol_rhs_row in kernels.h).

The solver appends the right-hand side(s) to the matrix as workspace rows R (and R + 1 for Jorion's vector of ones),
R = roundup(N, 8).  For N mod 32 in 1..24 these rows lie in the padding below Nr = roundup(N, 32) and, in the last
panel, inside the 32x32 diagonal block; otherwise R = Nr and the panels cover one more m-tile.  Both placements, with
one and two right-hand sides, on both solver kernels: chol_cluster_kernel is the default route of these small
launches, chol_solve_kernel runs in a child process with BP_CHOL_CLUSTER=0 (the knob is read once per process).
The reference and its bounds are those of tests/test_gpu_solver.py (tests/_solver_ref.py).
"""
import os
import subprocess
import sys

import numpy as np
import pytest

from tests import _solver_ref as ref
from tests.test_gpu_solver import GAMMA, V1, _check_solution, _engine, _pivot_problems, _sweep_problems

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

# N mod 32 = 1, 8, 20, 24, 1, 24, 20: the right-hand side sits in the padding rows (500 is the benchmark's N)
RHS_IN_PADDING = (33, 40, 52, 56, 257, 280, 500)
# N mod 32 = 25, 31, 0, 25, 0: it sits at row Nr
RHS_AT_NR = (57, 63, 64, 281, 288)
NS = RHS_IN_PADDING + RHS_AT_NR
# two right-hand sides: N mod 32 = 24, both rows fit below Nr; 25, neither does
JORION_NS = (56, 57, 280, 281)
BIG_RHS = 1e3
ROUTES = {"chol_cluster_kernel": None, "chol_solve_kernel": {"BP_CHOL_CLUSTER": "0"}}


def _big_rhs_problems(N):
    """Well-conditioned windows with a large right-hand side: in the last panel the right-hand-side row's own pivot,
    1 - |z in that panel|^2, is far below zero, and that must not be reported as a failed pivot of S."""
    rng = np.random.default_rng(80_000 + N)
    S = np.stack([ref.spd_with_kappa(N, 1e2, rng) for _ in range(2)])
    return S, BIG_RHS * rng.standard_normal((2, N))


def _jorion_problems(N):
    rng = np.random.default_rng(90_000 + N)
    probs = [ref.jorion_problem(N, rng) for _ in range(2)]
    return np.stack([p[0] for p in probs]), np.stack([p[1] for p in probs]), probs[0][2]


def _pack(res, prefix, out):
    for k in ("w1", "nu", "weights", "status"):
        out[f"{prefix}_{k}"] = res[k]
    out[f"{prefix}_scalars"] = res["scalars"]


def rhs_row_job(eng) -> dict:
    out = {}
    for N in NS:
        mats, rhs = _sweep_problems(N)
        _pack(eng.solve(np.stack([m[0] for m in mats]), rhs, jeffreys=True, risk_aversion=GAMMA), f"sweep{N}", out)
        S, b = _big_rhs_problems(N)
        _pack(eng.solve(S, b, jeffreys=True, risk_aversion=GAMMA), f"big{N}", out)
        bad, good, prhs, _ = _pivot_problems(N)
        n1 = np.full(len(prhs), 1e6)
        for tag, Sp in (("bad", bad), ("good", good)):
            _pack(eng.solve(Sp, prhs, jeffreys=False, n1=n1, risk_aversion=GAMMA), f"pivot{N}_{tag}", out)
    for N in JORION_NS:
        C, t, m = _jorion_problems(N)
        _pack(eng.solve(C, t, jorion=True, n_returns=m, risk_aversion=GAMMA), f"jorion{N}", out)
    return out


def _child_main(path):
    eng = _engine()
    np.savez(path, **rhs_row_job(eng))
    eng.close()


@pytest.fixture(scope="module")
def routes(tmp_path_factory):
    """{kernel: rhs_row_job results}"""
    res = {}
    d = tmp_path_factory.mktemp("rhs_row")
    for name, extra in ROUTES.items():
        if extra is None:
            eng = _engine()
            try:
                res[name] = rhs_row_job(eng)
            finally:
                eng.close()
            continue
        path = str(d / f"{name}.npz")
        env = dict(os.environ, PYTHONNOUSERSITE="1", **extra)
        r = subprocess.run([sys.executable, "-c", f"from tests.test_gpu_solver_rhs_row import _child_main; _child_main({path!r})"],
                           cwd=ROOT, env=env, capture_output=True, text=True, timeout=600)
        assert r.returncode == 0, f"child {extra} failed:\n{r.stdout}\n{r.stderr}"
        with np.load(path) as z:
            res[name] = {k: z[k] for k in z.files}
    return res


@pytest.mark.parametrize("route", list(ROUTES))
@pytest.mark.parametrize("N", NS)
def test_solution_against_refined_reference(routes, route, N):
    res = routes[route]
    mats, rhs = _sweep_problems(N)
    assert np.all(res[f"sweep{N}_status"] == 0), res[f"sweep{N}_status"]
    for i, (A, kappa, d) in enumerate(mats):
        _check_solution(A, rhs[i], res[f"sweep{N}_w1"][i], res[f"sweep{N}_scalars"][i, V1], kappa, f"{route} N={N} window {i}", d)
    S, b = _big_rhs_problems(N)
    assert np.all(res[f"big{N}_status"] == 0), f"{route} N={N}: the right-hand-side row was reported as a failed pivot"
    for i in range(len(S)):
        _check_solution(S[i], b[i], res[f"big{N}_w1"][i], res[f"big{N}_scalars"][i, V1], 1e2, f"{route} N={N} large rhs {i}")


@pytest.mark.parametrize("route", list(ROUTES))
@pytest.mark.parametrize("N", NS)
def test_pivot_status_exact(routes, route, N):
    res = routes[route]
    _, _, _, expected = _pivot_problems(N)
    got = res[f"pivot{N}_bad_status"]
    bad = np.nonzero(got != expected)[0]
    assert bad.size == 0, f"{route} N={N}: status {got[bad].tolist()} expected {expected[bad].tolist()}"
    assert np.all(res[f"pivot{N}_good_status"] == 0)
    healthy = expected == 0
    for k in ("w1", "nu", "weights", "scalars"):
        a, b = res[f"pivot{N}_bad_{k}"][healthy], res[f"pivot{N}_good_{k}"][healthy]
        assert np.array_equal(a, b), f"{route} N={N}: a failing window disturbed its neighbours' {k}"


@pytest.mark.parametrize("route", list(ROUTES))
@pytest.mark.parametrize("N", JORION_NS)
def test_jorion_two_rhs_rows(routes, route, N):
    res = routes[route]
    C, t, m = _jorion_problems(N)
    assert np.all(res[f"jorion{N}_status"] == 0)
    for i in range(len(C)):
        kappa = ref.kappa2(C[i])
        r = ref.jorion_reference(C[i], t[i], m, GAMMA, kappa)
        fwd = ref.forward_error(res[f"jorion{N}_w1"][i], r["y"].v)
        assert fwd <= ref.forward_bound(N, kappa), f"{route} N={N} window {i}: C^-1 t forward error {fwd:.3e}"
        for key in ("weights", "nu"):
            err = np.abs(res[f"jorion{N}_{key}"][i].astype(ref.LD) - r[key].v)
            assert np.all(err <= 2 * r[key].e), f"{route} N={N} window {i} {key}: max err/bound {float(np.max(err / r[key].e)):.2f}"


def test_kernels_bit_identical(routes):
    a, b = routes["chol_cluster_kernel"], routes["chol_solve_kernel"]
    assert set(a) == set(b)
    for k in a:
        x, y = a[k], b[k]
        if "_bad_" in k and not k.endswith("status"):       # what a failed factorisation leaves is no contract
            N = int(k[len("pivot"):k.index("_")])
            healthy = _pivot_problems(N)[3] == 0
            x, y = x[healthy], y[healthy]
        assert np.array_equal(x, y), f"{k} differs between the two solver kernels"


@pytest.mark.parametrize("N", (56, 500))
def test_poisoned_workspace_tail_is_ignored(N):
    """NaN left in the workspace by an all-NaN solve, padding rows included, must not reach a later solve whose
    right-hand sides live in those padding rows (R < Nr at these N)."""
    rng = np.random.default_rng(95_000 + N)
    S = np.stack([ref.spd_with_kappa(N, 1e4, rng) for _ in range(3)])
    rhs = rng.standard_normal((3, N))
    C, t, m = _jorion_problems(N)

    def run(eng, poison):
        out = []
        for solve in (lambda: eng.solve(S, rhs, jeffreys=True, risk_aversion=GAMMA),
                      lambda: eng.solve(C, t, jorion=True, n_returns=m, risk_aversion=GAMMA)):
            if poison:
                eng.solve(np.full((8, 513, 513), np.nan), np.full((8, 513), np.nan), jeffreys=True)
            out.append(solve())
        return out

    fresh_eng = _engine()
    try:
        fresh = run(fresh_eng, False)
    finally:
        fresh_eng.close()
    eng = _engine()
    try:
        got = run(eng, True)
    finally:
        eng.close()
    for what, g, f in zip(("jeffreys", "jorion"), got, fresh):
        for k in ("w1", "nu", "weights", "scalars", "status"):
            assert np.array_equal(g[k], f[k]), f"N={N} {what}: {k} depends on the workspace's old contents"
