#!/usr/bin/env python
"""The experiment the reference ships (portfolio_specs.py:54-62: top 50 of 500 by cap, monthly rebalancing, 250-week
window, conjugate HF-VIX VW) as bench.py's loop level runs it, on bench.py's 500-stock synthetic market, with the
windows of small asset sets stacked (``BayesEngine.set_stack_max_windows``, the default) and with one working market
and one batched call per asset set (``set_stack_max_windows(0)``).  One process: a warm-up pass of each, then the two
alternate; every pass records the wall-clock phases of ``backtest_portfolio`` (``timings``), the stacked windows and
calls and the kernel launches, and splits the weights phase into the pool upload, the working-market selections
(``select_market`` / ``select_windows`` / ``set_resampled``), the batched calls (which return with the weights in host
memory) and the host work between them.  The outputs of both routes are compared bit for bit, and their sha256 is
recorded so that two builds can be compared too.  The card's name and power limit are read in the same run.

    python tools/asset_sets_bench.py [--reps 5] [--lib PATH] [--out profiles/asset_sets_bench.json]

--lib loads another build of libbayes_portfolio.so (e.g. one of an earlier commit) in place of the package's.
"""
import argparse
import hashlib
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def card():
    import torch
    out = {"name": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30)
        out["nvidia_smi"] = q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else None
    except (OSError, subprocess.SubprocessError):
        out["nvidia_smi"] = None
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--n-assets", type=int, default=500)
    ap.add_argument("--windows", type=int, default=4150)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "asset_sets_bench.json"))
    ap.add_argument("--lib", help="libbayes_portfolio.so to load instead of the package's")
    args = ap.parse_args()
    import pandas as pd
    import bench
    from incorporating_different_sources_b200 import _lib
    from incorporating_different_sources_b200 import portfolio_calculations as pc
    if args.lib:
        _lib.LIB_PATH = os.path.abspath(args.lib)
    from incorporating_different_sources_b200.engine import BayesEngine

    mkt, _, _, d_idx = bench.make_workload(args, 0)
    md = mkt.market_data()
    ship = dict(weighting_strategy="conjugate_hf_vix_vw", size=50, risk_aversion=5, turnover_cost=15,
                rebalancing_frequency="monthly", rolling_window=250, rolling_window_frequency="weekly", mcm_scaling=1,
                display_name="Conjugate HF-VIX VW (shipped spec)")
    first = max(int(d_idx[0]), 1300)              # as bench.py: 250 complete weeks of history before the first rebalance
    start, end = pd.Timestamp(mkt.dates[first]), pd.Timestamp(mkt.dates[int(d_idx[-1])])
    eng = BayesEngine(0)
    spent = {}

    def timed(key, fn):
        def call(*a, **kw):
            t = time.perf_counter()
            try:
                return fn(*a, **kw)
            finally:
                spent[key] = spent.get(key, 0.0) + time.perf_counter() - t
        return call

    # the engine calls inside the weights phase, timed on the host (each of them ends in a synchronise or, for the
    # batched call, with the weights in host memory)
    upload, upload_timed = eng.upload_pool, timed("pool_upload_s", eng.upload_pool)
    eng.upload_pool = lambda prices, *a, **kw: (upload if prices is None else upload_timed)(prices, *a, **kw)
    for name in ("select_market", "select_windows", "set_resampled"):
        setattr(eng, name, timed("select_s", getattr(eng, name)))
    eng.conjugate = timed("batched_calls_s", eng.conjugate)

    def run(stack_max):
        eng.set_stack_max_windows(stack_max)
        tm = {}
        spent.clear()
        l0 = eng.launch_count
        t0 = time.perf_counter()
        res = pc.backtest_portfolio(ship, start, end, md, engine=eng, timings=tm)
        dt = time.perf_counter() - t0
        weights = dict(spent, host_planning_and_checks_s=tm["weights_s"] - sum(spent.values()))
        rec = dict(seconds=dt, launches=eng.launch_count - l0, weights_phase=weights, **tm)
        return rec, res

    routes = {"stacked": 15, "per_set": 0}
    passes = {k: [] for k in routes}
    outputs = {}
    for name, n in routes.items():                 # warm-up pass of each route (allocations, module loads)
        _, outputs[name] = run(n)
    for _ in range(args.reps):
        for name, n in routes.items():
            rec, _ = run(n)
            passes[name].append(rec)
    eng.set_stack_max_windows()
    identical = all(np.array_equal(outputs["stacked"][k].to_numpy(), outputs["per_set"][k].to_numpy(), equal_nan=True)
                    for k in outputs["stacked"])
    summary = {}
    for name, recs in passes.items():
        med = sorted(recs, key=lambda r: r["weights_s"])[len(recs) // 2]
        summary[name] = dict(median=med, weights_s_all=[r["weights_s"] for r in recs],
                             total_s_all=[r["total_s"] for r in recs], passes=recs)
    out = dict(tool="tools/asset_sets_bench.py", lib=os.path.relpath(_lib.LIB_PATH, ROOT), card=card(),
               spec="top 50 of 500 by cap, monthly rebalancing, 250-week window, conjugate HF-VIX VW, 7-day intraday look-back",
               market=dict(n_assets=args.n_assets, n_days=int(mkt.n_days), hf_rows=int(mkt.hf_prices.shape[0])), reps=args.reps,
               outputs_bit_identical=bool(identical), routes=summary,
               output_sha256={k: hashlib.sha256(np.ascontiguousarray(v.to_numpy()).tobytes()).hexdigest()
                              for k, v in outputs["per_set"].items()})
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(out, f, indent=1, default=float)
    print(json.dumps({k: dict(weights_s=v["median"]["weights_s"], total_s=v["median"]["total_s"],
                              weights_phase=v["median"]["weights_phase"], weights_s_all=v["weights_s_all"],
                              stacked_calls=v["median"].get("stacked_calls"), launches=v["median"]["launches"])
                      for k, v in summary.items()} | {"identical": identical, "card": out["card"]}))
    eng.close()


if __name__ == "__main__":
    main()
