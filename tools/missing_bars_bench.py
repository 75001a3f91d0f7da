#!/usr/bin/env python
"""Cost of missing intraday bars on the conjugate path (the C2 shape of bench.py: N = 500, n = 252).

A seeded fraction of the bars of ``--nan-cols`` held columns (illiquid names) is set to NaN; the return rows next to
each hole are dropped as the reference's dropna does (portfolio_calculations.py:314).  For every fraction the script
times one step -- the on-device log returns (bp_prepare_market) plus one conjugate batch with the weights read back --
and checks a sample of windows against the oracle with the dropna prior (tests/_dropna_ref.py).  Prints one JSON line
and writes it to ``--out`` when given.

    python tools/missing_bars_bench.py [--windows 1024] [--hf-days 7] [--fractions 0,0.001,0.01] [--out FILE]
"""
import argparse
import dataclasses
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n-assets", type=int, default=500)
    ap.add_argument("--windows", type=int, default=1024)
    ap.add_argument("--hf-days", type=int, default=7)
    ap.add_argument("--nan-cols", type=int, default=10)
    ap.add_argument("--fractions", default="0,0.001,0.01")
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--check", type=int, default=6, help="windows per fraction checked against the oracle")
    ap.add_argument("--seed", type=int, default=11)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()

    import torch
    from incorporating_different_sources_b200.engine import BayesEngine, upload_synthetic
    from incorporating_different_sources_b200.synthetic import generate_market
    from incorporating_different_sources_b200.windows import plan_daily_windows
    from oracle import bayes_oracle as bo
    from tests._dropna_ref import keep_mask, realized_covariance_dropna

    N, W = args.n_assets, args.windows
    first = 252 + (args.hf_days * 5) // 7 + 10
    base = generate_market(N, first + W, seed=args.seed)
    spec = dict(weighting_strategy="conjugate_hf_vix_vw", size=N, risk_aversion=5, turnover_cost=15,
                rebalancing_frequency="daily", rolling_window=252, rolling_window_frequency="daily", mcm_scaling=1)
    d_idx = list(range(first, first + W))
    batch = plan_daily_windows(spec, base.dates, d_idx, base.hf_ts, hf_lookback_days=args.hf_days)
    lo, hi = int(batch.hf_lo.min()), int(batch.hf_hi.max())
    rng = np.random.default_rng(args.seed)
    cols = rng.choice(N, size=args.nan_cols, replace=False)
    eng = BayesEngine(0)
    bo.realized_covariance = realized_covariance_dropna
    line = dict(tool="missing_bars_bench", gpu=torch.cuda.get_device_name(0), n_assets=N, windows=W,
                hf_days=args.hf_days, nan_cols=int(args.nan_cols), steps=args.steps, runs=[])
    for f in [float(x) for x in args.fractions.split(",")]:
        H = base.hf_prices.copy()
        sub = H[lo:hi, cols]
        sub[rng.random(sub.shape) < f] = np.nan
        H[lo:hi, cols] = sub
        mkt = dataclasses.replace(base, hf_prices=H)
        upload_synthetic(eng, mkt)
        for _ in range(args.warmup):
            eng.prepare_market()
            eng.conjugate(batch, outputs=("weights", "status"))
        eng.synchronize()
        t0 = time.perf_counter()
        for _ in range(args.steps):
            eng.prepare_market()
            got = eng.conjugate(batch, outputs=("weights", "scalars", "status"))
        eng.synchronize()
        ms = (time.perf_counter() - t0) * 1e3 / args.steps
        keep = keep_mask(H)
        span = batch.hf_hi - batch.hf_lo - 1
        m = got["scalars"][:, 6]
        err = 0.0
        for i in np.linspace(0, W - 1, args.check).astype(int):
            ref = bo.conjugate_window(spec, mkt, d_idx[i], np.arange(N), hf_lookback_days=args.hf_days)
            assert m[i] == ref["hf_returns"] == keep[batch.hf_lo[i] + 1:batch.hf_hi[i]].sum()
            err = max(err, float(np.max(np.abs(got["weights"][i] - ref["weights"])) / np.max(np.abs(ref["weights"]))))
        line["runs"].append(dict(nan_fraction=f, ms_per_step=ms, kept_rows_mean=float(np.mean(m / span)),
                                 windows_failed=int(np.count_nonzero(got["status"])),
                                 parity_max_rel_err=err, parity_windows=int(args.check)))
    eng.close()
    text = json.dumps(line)
    print(text)
    if args.out:
        with open(args.out, "w") as fh:
            fh.write(text + "\n")


if __name__ == "__main__":
    main()
