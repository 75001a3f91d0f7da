"""The Cholesky solver on its own (bp_solve_batched), against a reference far more accurate than float64.

Every launch route is pinned: chol_cluster_kernel with K = 8 / 4 / 2 CTAs per window, chol_solve_kernel with one wave
or a grid-stride loop, forced cluster sizes, one cluster looping over every window and several windows per CTA (the
last ones through the BP_CHOL_* knobs, read once per process, hence child processes), with one and two right-hand
sides.  The matrices and the reference live in tests/_solver_ref.py; the bounds are explained there.
"""
import os
import subprocess
import sys

import numpy as np
import pytest

from tests import _solver_ref as ref

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GAMMA = 3.0
V1 = 8                       # BP_SCAL_V1
JORION_SLOTS = dict(mu_g=0, lambda_hat=1, v_hat=2, q=4, one_vinv_one=5)

SWEEP_NS = [1, 2, 7, 8, 9, 15, 16, 17, 31, 32, 33, 63, 64, 65, 96, 127, 128, 129, 255, 257, 500, 511, 512, 513, 767,
            768, 769, 1023, 1536, 1537, 2048, 3072]
KAPPAS = (1e2, 1e8, 1e12)

# knob settings of the child processes: forced cluster sizes (0 = chol_solve_kernel only), one cluster looping over
# every window, several windows per CTA of chol_solve_kernel
CHILD_ENVS = [
    {"BP_CHOL_CLUSTER": "0"}, {"BP_CHOL_CLUSTER": "1"}, {"BP_CHOL_CLUSTER": "2"}, {"BP_CHOL_CLUSTER": "4"},
    {"BP_CHOL_CLUSTER": "8"}, {"BP_CHOL_CLUSTER": "8", "BP_CHOL_MAX_CLUSTERS": "1"},
    {"BP_CHOL_CLUSTER": "0", "BP_CHOL_CTAS_PER_SM": "1"},
]
PIVOT_NS = (8, 33, 100, 257, 500)


def _engine():
    from incorporating_different_sources_b200.engine import BayesEngine
    return BayesEngine(0, use_torch_stream=False)


@pytest.fixture(scope="module")
def engine():
    eng = _engine()
    yield eng
    eng.close()


def _check_solution(S, b, x, v1, kappa, what, d=None):
    """Backward error of x, forward error of x and v1 against the refined reference.  With d (the equilibration of a
    badly scaled S) the forward error is measured in the equilibrated variables d x, against kappa_2 of D^-1 S D^-1."""
    N = S.shape[0]
    eta = ref.backward_error(S, x, b)
    assert eta <= ref.eta_bound(N), f"{what}: backward error {eta:.3e} > {ref.eta_bound(N):.3e}"
    x_ref = ref.refined_solve(S, b)
    scale = np.ones(N) if d is None else d
    fwd = ref.forward_error(scale * x, scale.astype(ref.LD) * x_ref)
    bound = ref.forward_bound(N, kappa)
    assert fwd <= bound, f"{what}: forward error {fwd:.3e} > {bound:.3e} (kappa {kappa:.2e})"
    v1_ref = np.dot(np.asarray(b, dtype=ref.LD), x_ref)
    ev1 = float(abs(v1 - v1_ref) / abs(v1_ref))
    assert ev1 <= bound, f"{what}: v1 error {ev1:.3e} > {bound:.3e}"
    return x_ref, v1_ref


# ------------------------------------------------------------------------------------------- 1. shape sweep
def _sweep_problems(N):
    rng = np.random.default_rng(10_000 + N)
    mats = [(ref.spd_with_kappa(N, k, rng), k, None) for k in KAPPAS]
    if 2 <= N <= 1024:
        J, _ = ref.project_like(N, rng)
        mats.append((J, ref.kappa2(J), None))
        A, _ = ref.badly_scaled(mats[0][0], rng)
        H, d = ref.equilibrate(A)
        mats.append((A, ref.kappa2(H), d))
    rhs = rng.standard_normal((len(mats), N))
    return mats, rhs


@pytest.mark.parametrize("N", SWEEP_NS)
def test_shape_sweep_against_refined_reference(engine, N):
    mats, rhs = _sweep_problems(N)
    S = np.stack([m[0] for m in mats])
    jef = engine.solve(S, rhs, jeffreys=True, risk_aversion=GAMMA)
    assert np.all(jef["status"] == 0), jef["status"]
    v1_refs = []
    for i, (A, kappa, d) in enumerate(mats):
        _, v1_ref = _check_solution(A, rhs[i], jef["w1"][i], jef["scalars"][i, V1], kappa, f"N={N} window {i}", d)
        v1_refs.append(float(v1_ref))
    # conjugate scaling with n1 well above v1, so that n1 - v1 does not cancel
    n1 = 10.0 * np.abs(v1_refs) + N
    con = engine.solve(S, rhs, jeffreys=False, n1=n1, risk_aversion=GAMMA)
    assert np.all(con["status"] == 0)
    # the scaling is an epilogue: the factorisation and the solves are the same
    assert np.array_equal(con["w1"], jef["w1"])
    assert np.array_equal(con["scalars"][:, V1], jef["scalars"][:, V1])
    assert np.array_equal(con["scalars"][:, 1], n1)          # BP_SCAL_N1 is handed through


# ------------------------------------------------------------------------------------------- 5. epilogues
@pytest.mark.parametrize("N", [1, 33, 500, 1537, 3072])
def test_epilogues_bit_exact(engine, N):
    """nu and weights follow from the GPU's own w1 and v1 exactly as the reference writes them (:572-575, :836, :849)."""
    mats, rhs = _sweep_problems(N)
    S = np.stack([m[0] for m in mats[:3]])
    rhs = rhs[:3]
    jef = engine.solve(S, rhs, jeffreys=True, risk_aversion=GAMMA)
    assert np.array_equal(jef["nu"], jef["w1"])
    assert np.array_equal(jef["weights"], (1.0 / GAMMA) * jef["nu"])
    n1 = 10.0 * np.abs(jef["scalars"][:, V1]) + N
    con = engine.solve(S, rhs, jeffreys=False, n1=n1, risk_aversion=GAMMA)
    v1 = con["scalars"][:, V1]
    nu = con["w1"] * ((n1 + N + 2.0) / (n1 - v1))[:, None]
    assert np.array_equal(con["nu"], nu)
    assert np.array_equal(con["weights"], (1.0 / GAMMA) * nu)


@pytest.mark.parametrize("N", [31, 129, 768, 769, 1536])
def test_jorion_epilogue_against_oracle_formulas(engine, N):
    """Two right-hand sides (t and 1): N <= 768 runs chol_cluster_kernel<2>, larger N chol_solve_kernel<2>."""
    rng = np.random.default_rng(20_000 + N)
    probs = [ref.jorion_problem(N, rng) for _ in range(2)]
    C = np.stack([p[0] for p in probs])
    t = np.stack([p[1] for p in probs])
    m = probs[0][2]
    got = engine.solve(C, t, jorion=True, n_returns=m, risk_aversion=GAMMA)
    assert np.all(got["status"] == 0)
    for i, (Ci, ti, _) in enumerate(probs):
        kappa = ref.kappa2(Ci)
        r = ref.jorion_reference(Ci, ti, m, GAMMA, kappa)
        fwd = ref.forward_error(got["w1"][i], r["y"].v)
        assert fwd <= ref.forward_bound(N, kappa), f"window {i}: C^-1 t forward error {fwd:.3e}"
        for name, key in (("weights", "weights"), ("nu", "nu")):
            err = np.abs(got[key][i].astype(ref.LD) - r[name].v)
            assert np.all(err <= 2 * r[name].e), f"window {i} {name}: max err/bound {float(np.max(err / r[name].e)):.2f}"
        for name, slot in JORION_SLOTS.items():
            err = abs(ref.LD(got["scalars"][i, slot]) - r[name].v)
            assert err <= 2 * r[name].e, f"window {i} {name}: err {float(err):.3e} bound {float(r[name].e):.3e}"


# ------------------------------------------------------------------------------------------- 2./3. routes, pivots
def _route_sets(slots):
    """(N, W) of the route problem set: W = slots + 37 runs the grid-stride loop of chol_solve_kernel whole; N = 500
    keeps host memory bounded with W = slots / 4 + 5 (K = 2 whole)."""
    return [(40, slots + 37), (97, slots + 37), (500, slots // 4 + 5)]


def _route_problems(N, W):
    rng = np.random.default_rng(30_000 + N)
    S = np.empty((W, N, N))
    rhs = np.empty((W, N))
    for w in range(W):
        S[w], rhs[w] = ref.project_like(N, rng)
    return S, rhs


def _pivot_problems(N):
    """Failing windows interleaved with healthy ones; returns (S, S with every failing window made healthy, rhs,
    expected status)."""
    rng = np.random.default_rng(40_000 + N)
    cases = [("neg", [k]) for k in ref.pivot_columns(N)] + [("nan", [k]) for k in ref.pivot_columns(N)]
    two = ref.two_failures(N)
    if two:
        cases.append(("neg", list(two)))
    bad, good, status = [], [], []
    for kind, ks in cases:
        if kind == "neg":
            F = ref.failing_pivot_matrix(N, ks, rng)
        else:
            F = ref.healthy_matrix(N, rng)
            F[ks[0], ks[0]] = np.nan
        Hf = ref.healthy_matrix(N, rng)          # replaces F in the healthy batch
        Hn = ref.healthy_matrix(N, rng)          # the healthy neighbour
        bad += [F, Hn]
        good += [Hf, Hn]
        status += [min(ks) + 1, 0]
    rhs = rng.standard_normal((len(bad), N))
    return np.stack(bad), np.stack(good), rhs, np.array(status, dtype=np.int32)


def _jorion_route_problems(N):
    rng = np.random.default_rng(50_000 + N)
    probs = [ref.jorion_problem(N, rng) for _ in range(3)]
    return np.stack([p[0] for p in probs]), np.stack([p[1] for p in probs]), probs[0][2]


ROUTE_KEYS = ("w1", "nu", "weights", "v1", "status")


def _pack(res):
    return dict(w1=res["w1"], nu=res["nu"], weights=res["weights"], v1=res["scalars"][:, V1].copy(), status=res["status"])


def route_job(eng, slots: int) -> dict:
    """Everything that must not depend on the launch route, solved whole on this process's route.  ``slots`` (the
    default wave size) fixes the problem set: a child's knobs may change its own wave size."""
    out = {}
    for N, W in _route_sets(slots):
        S, rhs = _route_problems(N, W)
        for k, v in _pack(eng.solve(S, rhs, jeffreys=True, risk_aversion=GAMMA)).items():
            out[f"route{N}_{k}"] = v
    for N in PIVOT_NS:
        bad, good, rhs, _ = _pivot_problems(N)
        n1 = np.full(len(rhs), 1e6)
        for tag, S in (("bad", bad), ("good", good)):
            for k, v in _pack(eng.solve(S, rhs, jeffreys=False, n1=n1, risk_aversion=GAMMA)).items():
                out[f"pivot{N}_{tag}_{k}"] = v
    for N in (31, 129):
        C, t, m = _jorion_route_problems(N)
        res = eng.solve(C, t, jorion=True, n_returns=m, risk_aversion=GAMMA)
        for k, v in _pack(res).items():
            out[f"jorion{N}_{k}"] = v
        out[f"jorion{N}_scalars"] = res["scalars"]
    return out


def _child_main(path, slots):
    eng = _engine()
    np.savez(path, **route_job(eng, slots))
    eng.close()


@pytest.fixture(scope="module")
def routes(engine, tmp_path_factory):
    """{route name: route_job results}: this process (default thresholds) and one child process per knob setting."""
    slots = engine.solve_wave_windows()
    res = {"default": route_job(engine, slots)}
    d = tmp_path_factory.mktemp("routes")
    for i, extra in enumerate(CHILD_ENVS):
        path = str(d / f"child{i}.npz")
        env = dict(os.environ, PYTHONNOUSERSITE="1", **extra)
        r = subprocess.run([sys.executable, "-c", f"from tests.test_gpu_solver import _child_main; _child_main({path!r}, {slots})"],
                           cwd=ROOT, env=env, capture_output=True, text=True, timeout=600)
        assert r.returncode == 0, f"child {extra} failed:\n{r.stdout}\n{r.stderr}"
        with np.load(path) as z:
            res[" ".join(f"{k}={v}" for k, v in extra.items())] = {k: z[k] for k in z.files}
    return res


def _slices(W, slots):
    """Partitions of range(W) whose pieces land on K = 8, K = 4, K = 2, one chol_solve_kernel wave and the rest."""
    parts = []
    a = [slots // 8, slots // 4, slots // 2]
    if sum(a) < W:
        parts.append(a + [W - sum(a)])
    if slots // 2 + 1 < W:
        parts.append([slots // 2 + 1, W - slots // 2 - 1])
    if slots // 8 < W:
        parts.append([slots // 8, W - slots // 8])
    return parts


def test_routes_bit_identical_over_slices(engine):
    """The same windows split over launches of every size give the same bits as one launch of all of them."""
    slots = engine.solve_wave_windows()
    assert slots > 0
    for N, W in _route_sets(slots):
        S, rhs = _route_problems(N, W)
        whole = _pack(engine.solve(S, rhs, jeffreys=True, risk_aversion=GAMMA))
        assert np.all(whole["status"] == 0)
        for sizes in _slices(W, slots):
            pieces, w0 = [], 0
            for n in sizes:
                pieces.append(_pack(engine.solve(S[w0:w0 + n], rhs[w0:w0 + n], jeffreys=True, risk_aversion=GAMMA)))
                w0 += n
            for k in ROUTE_KEYS:
                cat = np.concatenate([p[k] for p in pieces])
                assert np.array_equal(cat, whole[k]), f"N={N} slices {sizes}: {k} differs from the whole launch"


def test_routes_bit_identical_across_kernels(routes):
    base = routes["default"]
    healthy = {N: _pivot_problems(N)[3] == 0 for N in PIVOT_NS}
    for name, res in routes.items():
        assert set(res) == set(base), name
        for k in base:
            a, b = res[k], base[k]
            if "_bad_" in k and not k.endswith("status"):       # what a failed factorisation leaves is no contract
                N = int(k[len("pivot"):k.index("_")])
                a, b = a[healthy[N]], b[healthy[N]]
            assert np.array_equal(a, b), f"route {name}: {k} differs from the default route"


def test_pivot_status_exact_on_every_route(routes):
    for name, res in routes.items():
        for N in PIVOT_NS:
            _, _, _, expected = _pivot_problems(N)
            got = res[f"pivot{N}_bad_status"]
            bad = np.nonzero(got != expected)[0]
            assert bad.size == 0, f"route {name} N={N}: status {got[bad].tolist()} expected {expected[bad].tolist()}"
            assert np.all(res[f"pivot{N}_good_status"] == 0)
            healthy = expected == 0
            for k in ("w1", "nu", "weights", "v1"):
                a, b = res[f"pivot{N}_bad_{k}"][healthy], res[f"pivot{N}_good_{k}"][healthy]
                assert np.array_equal(a, b), f"route {name} N={N}: a failing window disturbed its neighbours' {k}"


# ------------------------------------------------------------------------------------------- 4. lower triangle, padding
@pytest.mark.parametrize("N", [9, 33, 100, 257, 513, 1537])
def test_upper_triangle_is_not_read(engine, N):
    rng = np.random.default_rng(60_000 + N)
    S = np.stack([ref.spd_with_kappa(N, 1e4, rng) for _ in range(2)])
    rhs = rng.standard_normal((2, N))
    clean = engine.solve(S, rhs, jeffreys=True, risk_aversion=GAMMA)
    Sn = S.copy()
    iu = np.triu_indices(N, 1)
    Sn[:, iu[0], iu[1]] = np.nan
    poisoned = engine.solve(Sn, rhs, jeffreys=True, risk_aversion=GAMMA)
    for k in ("w1", "nu", "weights", "scalars", "status"):
        assert np.array_equal(poisoned[k], clean[k]), k


def _market_batches(eng):
    from incorporating_different_sources_b200.engine import upload_synthetic
    from incorporating_different_sources_b200.synthetic import generate_market
    from incorporating_different_sources_b200.windows import plan_daily_windows
    mkt = generate_market(10, 270, seed=7)
    spec = dict(weighting_strategy="conjugate_hf_vix_vw", size=10, risk_aversion=5, turnover_cost=15,
                rebalancing_frequency="daily", rolling_window=252, rolling_window_frequency="daily", mcm_scaling=1)
    d_idx = [260, 265, 269]
    upload_synthetic(eng, mkt)
    outs = ("weights", "nu", "w1", "scalars", "status")
    conj = eng.conjugate(plan_daily_windows(spec, mkt.dates, d_idx, mkt.hf_ts), outputs=outs)
    jspec = dict(spec, weighting_strategy="jeffreys", mcm_scaling=None)
    jeff = eng.jeffreys(plan_daily_windows(jspec, mkt.dates, d_idx, need_hf=False), outputs=outs)
    return conj, jeff


def test_poisoned_workspace_padding_is_ignored():
    """The workspace is shared by every entry point and never cleared: NaN left in it (padding rows and columns
    included) by an all-NaN solve must change no later result, of the solver or of the market pipeline."""
    eng = _engine()
    try:
        conj0, jeff0 = _market_batches(eng)
        eng.solve(np.full((8, 513, 513), np.nan), np.full((8, 513), np.nan), jeffreys=True)
        for N in (33, 100, 257):
            rng = np.random.default_rng(70_000 + N)
            S = np.stack([ref.spd_with_kappa(N, 1e6, rng) for _ in range(4)])
            rhs = rng.standard_normal((4, N))
            n1 = np.full(4, 1e5)
            got = eng.solve(S, rhs, jeffreys=False, n1=n1, risk_aversion=GAMMA)
            fresh_eng = _engine()
            try:
                fresh = fresh_eng.solve(S, rhs, jeffreys=False, n1=n1, risk_aversion=GAMMA)
            finally:
                fresh_eng.close()
            for k in ("w1", "nu", "weights", "scalars", "status"):
                assert np.array_equal(got[k], fresh[k]), f"N={N}: {k} depends on the workspace's old contents"
            eng.solve(np.full((8, 513, 513), np.nan), np.full((8, 513), np.nan), jeffreys=True)
        conj1, jeff1 = _market_batches(eng)
        for before, after, what in ((conj0, conj1, "conjugate"), (jeff0, jeff1, "jeffreys")):
            for k in before:
                assert np.array_equal(before[k], after[k]), f"{what} batch: {k} changed after the workspace was poisoned"
    finally:
        eng.close()


# ------------------------------------------------------------------------------------------- 6. limits
def _tiny_market(eng, N, D, rolling_window):
    from incorporating_different_sources_b200.windows import WindowBatch
    rng = np.random.default_rng(N)
    prices = 100.0 * np.exp(np.cumsum(rng.standard_normal((D, N)) * 0.01, axis=0))
    eng.upload_market(prices=prices, rf_row=np.zeros(D))
    return WindowBatch(rolling_window=rolling_window, day_row=np.array([D - 1], dtype=np.int32),
                       span_days=np.array([rolling_window + rolling_window // 2], dtype=np.int32), hf_lo=None, hf_hi=None,
                       risk_aversion=GAMMA)


def _assert_small_solve_works(eng):
    rng = np.random.default_rng(1)
    S = np.stack([ref.spd_with_kappa(40, 1e3, rng)])
    b = rng.standard_normal((1, 40))
    res = eng.solve(S, b, jeffreys=True)
    assert res["status"][0] == 0
    assert ref.backward_error(S[0], res["w1"][0], b[0]) <= ref.eta_bound(40)


def test_size_limits_fail_early_with_value_error():
    eng = _engine()
    try:
        N = 3073
        with pytest.raises(ValueError, match="at most 3072 assets"):
            eng.solve(np.zeros((1, N, N)), np.zeros((1, N)), jeffreys=True)
        _assert_small_solve_works(eng)
        batch = _tiny_market(eng, N, 12, 8)
        with pytest.raises(ValueError, match="at most 3072 assets"):
            eng.jeffreys(batch)
        _assert_small_solve_works(eng)
        with pytest.raises(ValueError, match="at most 3072 assets"):
            eng.dense_posterior(jeffreys=True, rolling_window=8, risk_aversion=GAMMA, T=np.eye(N), t=np.ones(N))
        _assert_small_solve_works(eng)
        N = 1537
        with pytest.raises(ValueError, match="at most 1536 assets"):
            eng.solve(np.zeros((1, N, N)), np.zeros((1, N)), jorion=True, n_returns=N + 10)
        _assert_small_solve_works(eng)
        batch = _tiny_market(eng, N, N + 20, N + 10)
        with pytest.raises(ValueError, match="at most 1536 assets"):
            eng.jorion(batch)
        _assert_small_solve_works(eng)
        # just inside the limits the same calls go through
        rng = np.random.default_rng(2)
        C, t, m = ref.jorion_problem(1536, rng)
        assert eng.solve(C[None], t[None], jorion=True, n_returns=m)["status"][0] == 0
    finally:
        eng.close()


def test_solve_rejects_outputs_it_does_not_produce(engine):
    S = np.eye(4)[None]
    b = np.ones((1, 4))
    for name in ("T", "S0", "S1", "t", "w0", "rhs"):
        with pytest.raises(ValueError, match="bp_solve_batched returns"):
            engine.solve(S, b, outputs=("weights", name))
    with pytest.raises(ValueError, match="needs n1"):
        engine.solve(S, b, jeffreys=False)
    with pytest.raises(ValueError, match="Jorion needs"):
        engine.solve(S, b, jorion=True, n_returns=6)
