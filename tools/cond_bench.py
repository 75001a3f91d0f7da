#!/usr/bin/env python
"""Cost of the condition estimate (bp_set_condition_estimate) on the C2 device-resident step of bench.py.

One step = on-device log returns + the 4,150 conjugate windows + the 4,150 Jeffreys windows at N = 500, weights and
status into device buffers (bench.py's ``value`` leg).  The step is timed with the estimate off and on, alternating in
this one process, ``--reps`` times each (CUDA events around each step); a second pass with per-stage timing gives the
``cond`` stage (anorm1 + rcond kernels) and the solve / chain stages, so that the Jeffreys cost of giving up the chain
(every window factorised while the estimate is on) is visible on its own.

Bytes read by the rcond kernel are counted, not measured: each application of A^-1 reads the lower triangle of the
factor twice (forward and back substitution), N (N + 1) / 2 * 8 bytes each, and the number of applications per window
comes from tests/_rcond_ref.py run on the S1 matrices of a sample of the conjugate windows (minus one: the kernel
solves dlacn2's last vector together with its first), applied to the Jeffreys windows too.  BP_RCOND_INFLIGHT_MB (read once per process) caps the windows in
flight of the rcond kernel; run the script once per setting.

    python tools/cond_bench.py [--reps 5] [--sample 24] [--out FILE]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def gpu_info():
    q = "name,power.limit,clocks.max.sm"
    try:
        r = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader"], capture_output=True, text=True,
                           timeout=30)
        return r.stdout.strip().splitlines()[0] if r.returncode == 0 and r.stdout.strip() else "unavailable"
    except Exception:
        return "unavailable"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n-assets", type=int, default=500)
    ap.add_argument("--windows", type=int, default=4150)
    ap.add_argument("--hf-days", type=int, default=7)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--sample", type=int, default=24, help="conjugate windows whose dlacn2 solve count is counted")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()

    import torch
    if not torch.cuda.is_available():
        raise SystemExit("cond_bench.py: no CUDA device")
    import bench
    from incorporating_different_sources_b200._lib import SCAL
    from incorporating_different_sources_b200.engine import BayesEngine
    from incorporating_different_sources_b200.windows import ffill_rows, plan_daily_windows, trim_intraday
    from tests import _rcond_ref as ref

    t_setup = time.perf_counter()
    mkt, conj, jeff, d_idx = bench.make_workload(argparse.Namespace(n_assets=args.n_assets, windows=args.windows), 0)
    N, W = args.n_assets, len(d_idx)
    cb = plan_daily_windows(conj, mkt.dates, d_idx, mkt.hf_ts, hf_lookback_days=args.hf_days)
    jb = plan_daily_windows(jeff, mkt.dates, d_idx, need_hf=False)
    lo, hi = trim_intraday(cb)
    dev = torch.device("cuda", 0)
    eng = BayesEngine(0)
    eng.upload_market(prices=mkt.prices, caps=mkt.caps, hf_prices=mkt.hf_prices[lo:hi], mcm=np.stack([mkt.vix, mkt.epu]),
                      rf_row=ffill_rows(mkt.dates, mkt.dates, mkt.rf))
    outs = {k: {"weights": torch.empty((W, N), dtype=torch.float64, device=dev),
                "status": torch.empty((W,), dtype=torch.int32, device=dev),
                "scalars": torch.empty((W, 12), dtype=torch.float64, device=dev)} for k in ("c", "j")}

    def step():
        eng.prepare_market()
        eng.conjugate(cb, outputs=("weights", "status", "scalars"), into=outs["c"])
        eng.jeffreys(jb, outputs=("weights", "status", "scalars"), into=outs["j"])

    def timed(flag):
        eng.set_condition_estimate(flag)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        step()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1)

    setup_s = time.perf_counter() - t_setup
    for _ in range(args.warmup):
        timed(False)
        timed(True)
    ms = {False: [], True: []}
    for _ in range(args.reps):
        for flag in (False, True):
            ms[flag].append(timed(flag))
    # outputs other than the estimate: the same bits
    eng.set_condition_estimate(False)
    step()
    ref_w = {k: outs[k]["weights"].clone() for k in outs}
    eng.set_condition_estimate(True)
    step()
    torch.cuda.synchronize()
    # the Jeffreys windows are chained with the estimate off: compare with the per-window path there
    same_conj = bool(torch.equal(ref_w["c"], outs["c"]["weights"]))
    rcond_c = outs["c"]["scalars"][:, SCAL["rcond"]].cpu().numpy()
    rcond_j = outs["j"]["scalars"][:, SCAL["rcond"]].cpu().numpy()

    stages = {}
    for flag in (False, True):
        eng.set_condition_estimate(flag)
        eng.set_stage_timing(True)
        eng.stage_times()
        eng.solve_work()
        for _ in range(args.reps):
            step()
        st = eng.stage_times()
        sw = eng.solve_work()
        eng.set_stage_timing(False)
        stages["on" if flag else "off"] = {"stages_ms_per_step": {k: v["ms"] / args.reps for k, v in st.items()},
                                           "launches_per_step": {k: v["launches"] / args.reps for k, v in st.items()},
                                           "windows_factorised_per_step": sw["factored"] / args.reps,
                                           "windows_chained_per_step": sw["chained"] / args.reps}
    eng.set_condition_estimate(False)

    # dlacn2 applications of A^-1 on a sample of conjugate windows (S1 of the same windows), CPU
    pick = np.linspace(0, W - 1, args.sample).astype(int)
    sb = plan_daily_windows(conj, mkt.dates, [int(d_idx[i]) for i in pick], mkt.hf_ts, hf_lookback_days=args.hf_days)
    sb.hf_lo, sb.hf_hi = sb.hf_lo - lo, sb.hf_hi - lo
    S1 = eng.conjugate(sb, outputs=("S1",))["S1"]
    solves = []
    for A in S1:
        r, k = ref.rcond(np.linalg.cholesky(A), ref.anorm1(A))
        solves.append(k)
    passes = float(np.mean(solves)) - 1.0                  # the kernel merges dlacn2's last solve into its first
    tri = N * (N + 1) / 2 * 8
    on = stages["on"]
    rcond_bytes = W * 2 * (passes * 2 * tri)               # conjugate + Jeffreys windows, fwd + back per pass
    norm_bytes = 2 * W * 2 * tri                            # column pass + row pass over the triangle
    cond_ms = on["stages_ms_per_step"]["cond"]
    line = dict(
        tool="cond_bench", gpu=gpu_info(), torch_device=torch.cuda.get_device_name(0),
        rcond_inflight_mb=os.environ.get("BP_RCOND_INFLIGHT_MB", "unset (one CTA per window)"),
        n_assets=N, windows_per_prior=W, hf_days=args.hf_days, reps=args.reps, setup_s=round(setup_s, 1),
        step_ms_off=ms[False], step_ms_on=ms[True],
        step_ms_off_median=float(np.median(ms[False])), step_ms_on_median=float(np.median(ms[True])),
        stages=stages, cond_stage_ms=cond_ms,
        solves_per_window_dpocon_mean=float(np.mean(solves)), solves_per_window_dpocon_max=int(np.max(solves)),
        rcond_passes_per_window_mean=passes,
        rcond_bytes_counted=rcond_bytes, norm_bytes_counted=norm_bytes,
        cond_stage_gbs_counted=(rcond_bytes + norm_bytes) / (cond_ms * 1e-3) / 1e9 if cond_ms > 0 else None,
        conj_weights_same_bits=same_conj,
        rcond_conj_min_median_max=[float(np.min(rcond_c)), float(np.median(rcond_c)), float(np.max(rcond_c))],
        rcond_jeff_min_median_max=[float(np.min(rcond_j)), float(np.median(rcond_j)), float(np.max(rcond_j))],
    )
    s = json.dumps(line)
    print(s)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(s + "\n")
    eng.close()


if __name__ == "__main__":
    main()
