"""Route fingerprint of the batched driver: for a fixed, seeded matrix of small cases that covers every route the
driver can take, what each call did -- launches in total and per stage (stage timing on), the Gram and solve work
counters, the return code and message -- and a sha256 of every output array.  Two builds that issue the same device
work in the same order give equal fingerprints.  Every case runs twice; a case whose output hashes differ between its
two runs is flagged ("deterministic": false), and a case whose second run differs in anything also records it
("second_run").

    python tools/driver_fingerprint.py [--lib PATH] --out FILE.json

--lib loads another build of libbayes_portfolio.so (e.g. one of an earlier commit) in place of the package's.
The working-market selections from the pool (select_market, select_windows) are cases of their own too: their launch
counts are the gathers and the daily log returns.
"""
import argparse
import hashlib
import json
import os
import re
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

ALL = ("T", "S0", "S1", "t", "w0", "rhs", "scalars", "weights", "nu", "w1", "status")
SOLVE = ("weights", "nu", "w1", "status", "t", "rhs", "scalars")
NO_REUSE = 2 ** 31 - 1


def _spec(N, rw, strategy="conjugate_hf_vix_vw", freq="daily", risk_aversion=5):
    return dict(weighting_strategy=strategy, size=N, risk_aversion=risk_aversion, rolling_window=rw,
                rolling_window_frequency=freq, mcm_scaling=1)


def _sha(v):
    if hasattr(v, "detach"):
        v = v.detach().cpu().numpy()
    return hashlib.sha256(np.ascontiguousarray(v).tobytes()).hexdigest()


def _hashes(out):
    if out is None:
        return {}
    if isinstance(out, tuple):
        out = {f"out{i}": v for i, v in enumerate(out)}
    return {k: _sha(v) for k, v in sorted(out.items()) if v is not None}


class Runner:
    def __init__(self, eng):
        self.eng = eng
        self.cases = {}

    def run(self, name, setup, call, teardown=None):
        from incorporating_different_sources_b200.engine import BayesPortfolioError
        eng = self.eng
        runs = []
        for _ in range(2):
            if setup:
                setup()
            eng.synchronize()
            eng.stage_times()
            eng.gram_work()
            eng.solve_work()
            l0 = eng.launch_count
            rc, msg, out = 0, "", None
            try:
                out = call()
                eng.synchronize()
            except ValueError as e:
                rc, msg = 1, str(e)
            except BayesPortfolioError as e:
                m = re.match(r"libbayes_portfolio error (\d+): (.*)", str(e), re.S)
                rc, msg = (int(m.group(1)), m.group(2)) if m else (-1, str(e))
            launches = eng.launch_count - l0
            stages = {k: v["launches"] for k, v in eng.stage_times().items()}
            runs.append(dict(rc=rc, msg=msg, launches=launches, stage_launches=stages, gram_work=eng.gram_work(),
                             solve_work=eng.solve_work(), hashes=_hashes(out)))
            if teardown:
                teardown()
        rec = dict(runs[0])
        rec["deterministic"] = runs[0]["hashes"] == runs[1]["hashes"]
        # the first call after an upload or a market selection also computes the intraday log returns (one launch)
        if runs[0] != runs[1]:
            rec["second_run"] = runs[1]
        self.cases[name] = rec
        print(f"{name:36s} rc={rec['rc']} launches={rec['launches']:5d} det={rec['deterministic']}", flush=True)


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n\n")[0])
    ap.add_argument("--lib", help="libbayes_portfolio.so to load instead of the package's")
    ap.add_argument("--out", required=True)
    args = ap.parse_args()
    from incorporating_different_sources_b200 import _lib
    if args.lib:
        _lib.LIB_PATH = os.path.abspath(args.lib)
    import torch
    from incorporating_different_sources_b200.backtest import _set_slice
    from incorporating_different_sources_b200.engine import BayesEngine, upload_synthetic
    from incorporating_different_sources_b200.synthetic import generate_market
    from incorporating_different_sources_b200.windows import (ffill_rows, plan_daily_windows, plan_weekly_windows,
                                                             stack_windows)

    eng = BayesEngine(0)
    eng.set_stage_timing(True)
    R = Runner(eng)
    N = 24

    # ---- conjugate on a daily market: every Gram route, chunking, output kinds
    mkt = generate_market(N, 330, seed=11)
    upload_synthetic(eng, mkt)
    conj = lambda b, outs=ALL, **kw: (lambda: eng.conjugate(b, outputs=outs, **kw))      # noqa: E731
    consec = plan_daily_windows(_spec(N, 60), mkt.dates, range(60, 110), mkt.hf_ts, hf_lookback_days=7)
    every3 = plan_daily_windows(_spec(N, 60), mkt.dates, range(60, 330, 3), mkt.hf_ts, hf_lookback_days=7)
    long_rw = plan_daily_windows(_spec(N, 200), mkt.dates, range(200, 250), mkt.hf_ts, hf_lookback_days=1)
    presum = plan_daily_windows(_spec(N, 60), mkt.dates, range(60, 110), mkt.hf_ts, hf_lookback_days=31)

    def reuse(n):
        return lambda: eng.set_reuse_min_windows(n)
    R.run("conj_from_scratch", reuse(NO_REUSE), conj(consec), reuse(32))
    R.run("conj_daily_block_reuse", None, conj(long_rw))
    R.run("conj_intraday_blocks", None, conj(every3))
    R.run("conj_inner_day_blocks", None, conj(consec))
    R.run("conj_presummed_day_blocks", None, conj(presum))
    R.run("conj_presummed_solve_only", None, conj(presum, ("weights", "status", "rhs", "scalars")))
    R.run("conj_presummed_moments", None, lambda: eng.moments(presum, outputs=("t", "w0", "rhs", "scalars")))
    R.run("conj_chunked", lambda: eng.set_workspace_limit(256 << 10), conj(consec),
          lambda: eng.set_workspace_limit(24 << 30))
    R.run("conj_chunked_presummed", lambda: eng.set_workspace_limit(256 << 10), conj(presum),
          lambda: eng.set_workspace_limit(24 << 30))
    R.run("conj_device_outputs", None, conj(consec, device_out=True))

    def async_out():
        W = consec.n_windows
        bufs = {"weights": torch.zeros(W, N, dtype=torch.float64).pin_memory().numpy(),
                "status": torch.ones(W, dtype=torch.int32).pin_memory().numpy()}
        eng.set_async_outputs(True)
        try:
            eng.conjugate(consec, outputs=("weights", "status"), into=bufs)
            eng.jeffreys(plan_daily_windows(_spec(N, 60, "jeffreys"), mkt.dates, range(60, 110), need_hf=False),
                         outputs=("weights",))
            eng.synchronize()
        finally:
            eng.set_async_outputs(False)
        return bufs
    R.run("conj_async_outputs", None, async_out)

    # ---- Jeffreys, estimators, moments on the same market
    jb = plan_daily_windows(_spec(N, 60, "jeffreys"), mkt.dates, range(60, 110), need_hf=False)
    jb3 = plan_daily_windows(_spec(N, 60, "jeffreys"), mkt.dates, range(60, 330, 3), need_hf=False)
    R.run("jeffreys_plain", None, lambda: eng.jeffreys(jb3, outputs=("weights", "nu", "w1", "status", "t", "rhs", "scalars")))
    R.run("jeffreys_chain", None, lambda: eng.jeffreys(jb, outputs=("weights", "nu", "w1", "status", "scalars")))
    R.run("jeffreys_chain_off_by_cond", lambda: eng.set_condition_estimate(True),
          lambda: eng.jeffreys(jb, outputs=("weights", "nu", "w1", "status", "scalars")),
          lambda: eng.set_condition_estimate(False))
    R.run("jeffreys_with_S1", None, lambda: eng.jeffreys(jb, outputs=("weights", "S1", "T", "status")))
    R.run("jorion", None, lambda: eng.jorion(jb, outputs=SOLVE + ("S1",)))
    R.run("jorion_chain", None, lambda: eng.jorion(jb, outputs=("weights", "status", "scalars")))
    R.run("shrinkage", None, lambda: eng.shrinkage(jb, outputs=SOLVE + ("S1",)))
    R.run("stats", None, lambda: eng.stats(jb))
    R.run("hf_cov", None, lambda: eng.hf_cov(consec))
    R.run("moments_conjugate", None, lambda: eng.moments(consec, outputs=("T", "S0", "S1", "t", "w0", "rhs", "scalars")))
    R.run("moments_jeffreys", None, lambda: eng.moments(jb, outputs=("T", "S1", "t", "rhs", "scalars"), jeffreys=True))

    # ---- solve entry points
    rng = np.random.default_rng(5)
    W = 20
    X = rng.standard_normal((W, 80, N))
    S = np.einsum("wki,wkj->wij", X, X)
    rhs = rng.standard_normal((W, N))
    R.run("solve_conjugate", None, lambda: eng.solve(S, rhs, jeffreys=False, n1=np.full(W, 90.0)))
    R.run("solve_jeffreys", None, lambda: eng.solve(S, rhs))
    R.run("solve_jorion", None, lambda: eng.solve(S, rhs, jorion=True, n_returns=79))
    R.run("solve_chunked", lambda: eng.set_workspace_limit(200 << 10), lambda: eng.solve(S, rhs),
          lambda: eng.set_workspace_limit(24 << 30))
    R.run("dense_posterior_jeffreys", None,
          lambda: eng.dense_posterior(jeffreys=True, rolling_window=81, risk_aversion=5, T=S[0], t=rhs[0]))
    R.run("dense_posterior_conjugate", None,
          lambda: eng.dense_posterior(jeffreys=False, rolling_window=81, risk_aversion=5, T=S[0], t=rhs[0], S0=S[1] / 80,
                                      w0=np.full(N, 1.0 / N), n0=30.0))

    # ---- error paths: the call's own arguments, and an invalid batch that also has them wrong
    bad_gamma = plan_daily_windows(_spec(N, 60, risk_aversion=0), mkt.dates, range(60, 110), mkt.hf_ts, hf_lookback_days=7)
    jb_gamma0 = plan_daily_windows(_spec(N, 60, "jeffreys", risk_aversion=0), mkt.dates, range(60, 110), need_hf=False)
    short = plan_daily_windows(_spec(N, 26, "jorion"), mkt.dates, range(60, 110), need_hf=False)
    R.run("error_conjugate_risk_aversion_0", None, conj(bad_gamma, ("weights",)))
    R.run("jeffreys_risk_aversion_0_unchecked", None, lambda: eng.jeffreys(jb_gamma0, outputs=("status",)))
    R.run("error_jorion_T_N_2", None, lambda: eng.jorion(short, outputs=("weights",)))
    invalid = plan_daily_windows(_spec(N, 60, risk_aversion=0), mkt.dates, range(60, 110), mkt.hf_ts, hf_lookback_days=7)
    invalid.day_row = np.array(invalid.day_row, dtype=np.int32)
    invalid.day_row[3] = 5
    R.run("error_invalid_batch_first", None, conj(invalid, ("weights",)))

    # ---- weekly (resampled) windows
    wm = generate_market(20, 460, seed=801)
    upload_synthetic(eng, wm)
    rows, wk = plan_weekly_windows(_spec(20, 60, freq="weekly", strategy="conjugate_hf_epu_vw"), wm.dates,
                                   list(range(430, 460)), wm.dates, wm.rf, np.stack([wm.vix, wm.epu]), wm.hf_ts)
    eng.set_resampled(rows)
    R.run("conj_weekly", None, lambda: eng.conjugate(wk, outputs=ALL))

    # ---- one asset set's working market gathered from the pool (select_market), sliced as backtest's per-set route
    # cuts it: the selection on its own, then a conjugate call with block reuse and a Jeffreys call with the chain
    pm = generate_market(40, 200, seed=31)
    eng.upload_pool(prices=pm.prices, rf_row=ffill_rows(pm.dates, pm.dates, pm.rf), caps=pm.caps, hf_prices=pm.hf_prices)
    pcols = np.random.default_rng(3).permutation(40)[:N]
    pb = plan_daily_windows(_spec(N, 60), pm.dates, list(range(100, 140)), pm.hf_ts, hf_lookback_days=7)
    psl = _set_slice(pb, pm.n_days, len(pm.hf_ts))
    pb.prior_n = np.full(pb.n_windows, 30.0)
    jpb = plan_daily_windows(_spec(N, 60, "jeffreys"), pm.dates, list(range(100, 140)), need_hf=False)
    jsl = _set_slice(jpb, pm.n_days, len(pm.hf_ts))
    R.run("select_market", None, lambda: eng.select_market(pcols, *psl))
    R.run("conj_pool_block_reuse", lambda: eng.select_market(pcols, *psl), conj(pb))
    R.run("jeffreys_pool_chain", lambda: eng.select_market(pcols, *jsl),
          lambda: eng.jeffreys(jpb, outputs=("weights", "nu", "w1", "status", "scalars")))

    # ---- stacked working market (select_windows)
    sb = plan_daily_windows(_spec(N, 60), pm.dates, list(range(100, 140, 2)), pm.hf_ts, hf_lookback_days=7)
    stk = stack_windows(sb, None)
    cols = np.stack([np.sort(np.random.default_rng(i).choice(40, N, replace=False)) for i in range(sb.n_windows)])
    R.run("select_windows", None, lambda: eng.select_windows(cols, np.stack([stk.day_lo, stk.day_hi], axis=1),
                                                             np.stack([stk.hf_lo, stk.hf_hi], axis=1)))
    stk.batch.prior_n = np.full(sb.n_windows, 30.0)
    R.run("conj_stacked", None, lambda: eng.conjugate(stk.batch, outputs=ALL))
    jstk = stack_windows(plan_daily_windows(_spec(N, 60, "jeffreys"), pm.dates, list(range(100, 140)), need_hf=False), None)
    eng.select_windows(np.repeat(cols[:1], 40, axis=0), np.stack([jstk.day_lo, jstk.day_hi], axis=1))
    R.run("jeffreys_stacked", None, lambda: eng.jeffreys(jstk.batch, outputs=("weights", "status", "scalars")))
    eng.upload_pool(None, None)

    # ---- pipelined against a segmented asynchronous intraday upload
    qm = generate_market(40, 600, seed=23)
    arrays = dict(prices=qm.prices, caps=qm.caps, hf_prices=qm.hf_prices, mcm=np.stack([qm.vix, qm.epu]),
                  rf_row=ffill_rows(qm.dates, qm.dates, qm.rf))
    pinned = {k: torch.from_numpy(np.ascontiguousarray(v)).pin_memory().numpy() for k, v in arrays.items()}
    qb = plan_daily_windows(_spec(40, 60), qm.dates, list(range(60, 600)), qm.hf_ts, hf_lookback_days=7)
    eng.upload_market(**arrays)
    pipe = ("weights", "scalars", "status", "w1")
    eng.set_upload_pipeline(8, 0)
    fractions = {"geometric": None, "waves": eng.plan_upload_fractions(qb, qm.hf_prices.shape[0])}
    for fname, fr in fractions.items():
        for outs in (pipe, pipe + ("S1",)):
            def setup(fr=fr):
                eng.set_upload_fractions(fr)
                eng.upload_market(**pinned, async_copy=True)
            R.run(f"conj_pipelined_{fname}" + ("_S1" if "S1" in outs else ""), setup, conj(qb, outs))
    eng.set_upload_fractions(None)
    R.run("conj_pipelined_device_S1", lambda: eng.upload_market(**pinned, async_copy=True),
          conj(qb, pipe + ("S1",), device_out=True))
    R.run("conj_async_upload_T_waits", lambda: eng.upload_market(**pinned, async_copy=True), conj(qb, ("weights", "T")))
    eng.set_upload_pipeline()
    eng.close()

    out = dict(lib=os.path.relpath(_lib.LIB_PATH, ROOT), device=torch.cuda.get_device_name(0), cases=R.cases)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(out, f, indent=1, sort_keys=True)
    bad = [k for k, v in R.cases.items() if not v["deterministic"]]
    print(f"{len(R.cases)} cases, nondeterministic: {bad or 'none'} -> {args.out}")


if __name__ == "__main__":
    main()
