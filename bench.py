#!/usr/bin/env python
"""Benchmark of the rolling-window Bayesian tangency-weight hot path (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]

Workload (BASELINE.json configs[1], "C2"): one full daily-rebalance backtest, 4,150 rebalance dates,
N = 500 synthetic assets, conjugate (VIX-scaled HF prior) + Jeffreys priors = 8,300 windows per step:
  * conjugate: 252-day daily window + 5-minute intraday prior over the reference's 7-calendar-day
    look-back (389 HF returns).  The reference's own 1-day look-back is rank deficient at N = 500
    (SURVEY F6: rank <= 76 + 251 < 500), so the well-posed look-back from its table (:299-304) is used,
    which the reference itself reaches through ``conjugate_prior_S_df=``;
  * Jeffreys: rolling_window = 1008 (n-1 >= N is required for T - tt'/n to be non-singular).
A "step" is one pass of the whole path over that backtest: log returns, per-window reductions and
prior scalars, batched Gram (DMMA), batched Cholesky solve, weights.  ``value`` times it with the
prices already resident in HBM; ``e2e`` times the public host-buffer API including the host->device
copy of the market and the device->host read of the weights.  N > 1 GPUs: weak scaling, one
independent synthetic path per rank (BASELINE configs[4]), weights all-gathered with NCCL.

``--impl reference`` times the UNMODIFIED reference (its sources staged under baseline/_ref/src by
``__graft_entry__.build()``, imported through oracle/ref_import.py, driven one window at a time by
oracle/ref_runner.py exactly as SURVEY 8(c)/(d) prescribes) on a bounded sample of the same windows with
every host core (level L0-mp of BASELINE.md section 3: one worker process per core, one BLAS thread each);
L0 (one process, default BLAS threads), L1 (``backtest_portfolio`` as shipped) and the NumPy port
(oracle/bayes_oracle.py) are reported beside it.  Only if the staged sources are missing does the arm fall
back to the port (``kind: "port"``).
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "posterior tangency-weight windows/sec at N=500"
UNIT = "windows/s"
DUMP_LIMIT_BYTES = 64 << 20


# ----------------------------------------------------------------------------- workload
def make_specs(n_assets):
    conj = dict(weighting_strategy="conjugate_hf_vix_vw", size=n_assets, risk_aversion=5, turnover_cost=15,
                rebalancing_frequency="daily", rolling_window=252, rolling_window_frequency="daily",
                mcm_scaling=1, display_name="Conjugate HF-VIX VW")
    jeff = dict(conj, weighting_strategy="jeffreys", mcm_scaling=None, rolling_window=max(1008, 2 * n_assets + 8),
                display_name="Jeffreys")
    return conj, jeff


def make_workload(args, path):
    from incorporating_different_sources_b200.synthetic import generate_market
    conj, jeff = make_specs(args.n_assets)
    n_long = jeff["rolling_window"]
    n_days = n_long + args.windows - 1
    start = str(np.busday_offset(np.datetime64("2007-01-01"), -(n_long - 1), roll="forward"))
    mkt = generate_market(args.n_assets, n_days, seed=1000 * path + 2, start=start)
    d_idx = np.arange(n_long - 1, n_days)
    return mkt, conj, jeff, d_idx


def config_dict(args, n_gpus, conj, jeff, hf_days):
    return {
        "workload": "C2: full daily-rebalance backtest, conjugate(VIX)+Jeffreys, synthetic S&P-500-sized universe",
        "n_assets": args.n_assets, "rebalance_dates": args.windows, "windows_per_step_per_gpu": 2 * args.windows,
        "conjugate": {"rolling_window": conj["rolling_window"], "hf_lookback_calendar_days": hf_days,
                      "hf_bar_minutes": 5, "prior": "vw", "mcm": "VIX",
                      "hf_lookback_note": "SURVEY 8(d) asks for an injected look-back >= 5 days at N=500 (the reference's own "
                                          "1-day window is rank deficient, F6); 7 calendar days is the shortest one in the "
                                          "reference's table (:299-304); --hf-days 366 (252 trading days) costs 1.1x this step "
                                          "(profiles/r2*_bench_hf366.json)"},
        "jeffreys": {"rolling_window": jeff["rolling_window"]},
        "sharding": f"{n_gpus} independent synthetic path(s), one per GPU; weights all-gathered (NCCL)" if n_gpus > 1
        else "single GPU, one path",
        "cache": "inputs larger than L2 (1.3 GB intraday prices, 8.8 GB workspace); no flush needed",
    }


def intraday_config(mkt, conj, d_idx, hf_days):
    """Which intraday rows belong to the workload (same fields in both arms' ``config``)."""
    from incorporating_different_sources_b200.windows import plan_daily_windows, trim_intraday
    lo, hi = trim_intraday(plan_daily_windows(conj, mkt.dates, d_idx, mkt.hf_ts, hf_lookback_days=hf_days))
    return dict(intraday_rows_uploaded=int(hi - lo), intraday_rows_in_market=int(mkt.hf_prices.shape[0]),
                intraday_note="bars before the first window's look-back (history only the daily windows need) are "
                              "read by no window and are not uploaded")


def dump_outputs(out_dir, arrays):
    """Write each array as ``out_dir/<name>.npy`` in float64, so that two builds can be compared output for output.
    Past DUMP_LIMIT_BYTES in all, every 2-D array (one row per window, all with the same rows) keeps the same seeded
    sample of rows, so runs with the same arguments write the same rows."""
    arrays = {k: np.asarray(v, dtype=np.float64) for k, v in arrays.items()}
    total = sum(a.nbytes for a in arrays.values())
    if total > DUMP_LIMIT_BYTES:
        rows2d = [a for a in arrays.values() if a.ndim == 2]
        row_bytes = sum(a.shape[1] * a.itemsize for a in rows2d)
        other = total - sum(a.nbytes for a in rows2d)
        keep = max(1, (DUMP_LIMIT_BYTES - other) // row_bytes)
        rows = np.sort(np.random.default_rng(0).choice(rows2d[0].shape[0], keep, replace=False))
        arrays = {k: a[rows] if a.ndim == 2 else a for k, a in arrays.items()}
        print(f"bench.py: outputs exceed {DUMP_LIMIT_BYTES >> 20} MB, writing a seeded sample of {keep} rows",
              file=sys.stderr)
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


# ----------------------------------------------------------------------------- clocks
class ClockSampler:
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index = index
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100", "-i",
                 str(self.index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons, pw = [], [], set(), []
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0])); mx.append(float(f[1])); pw.append(float(f[2]))
            except ValueError:
                continue
            for nm, v in zip(names, f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        return {"sm_mhz": float(np.median(sm)), "sm_max_mhz": float(max(mx)), "power_w_max": float(max(pw)),
                "samples": len(sm), "reasons": sorted(reasons)}


# ----------------------------------------------------------------------------- flops / bytes
def algorithmic_work(N, W, n_c, m_hf, n_j):
    """SURVEY §8(d) conventions: full-matrix DGEMM flops; compulsory bytes."""
    gram_conj = 2.0 * N * N * ((n_c - 1) + m_hf)
    gram_jeff = 2.0 * N * N * (n_j - 1)
    chol = N ** 3 / 3.0 + 4.0 * N * N
    nt = (N + 127) // 128
    tile_elems = nt * (nt + 1) // 2 * 128 * 128
    kx = lambda k: (k + 7) // 8 * 8                      # the kernel skips k-groups of 8 past the window end
    executed = 2.0 * tile_elems * (kx(n_c - 1) + kx(m_hf) + kx(n_j - 1))
    syrk_min = 1.0 * N * (N + 1) * ((n_c - 1) + m_hf + (n_j - 1))
    return {
        "gram_flops_executed": W * executed,
        "gram_flops_syrk_min": W * syrk_min,
        "gram_flops": W * (gram_conj + gram_jeff),
        "solve_flops": 2 * W * chol,
        "solve_bytes": 2 * W * (8.0 * N * N + 16.0 * N),
        "prep_bytes": W * 8.0 * N * ((n_c - 1) + 2 * m_hf + (n_j - 1)),
    }


# ----------------------------------------------------------------------------- reference arm
_G = {}


def _ref_window(job):
    """One window on one worker: the unmodified reference (kind 'reference') or the NumPy port (kind 'port').
    Returns the weights in ticker order."""
    kind, d = job
    mkt, conj, jeff, cols, hf_days = _G["mkt"], _G["conj"], _G["jeff"], _G["cols"], _G["hf_days"]
    if _G["impl"] == "reference":
        from oracle import ref_runner as rr
        pc = _G["pc"]
        if kind == 0:
            df = rr.conjugate_window(pc, conj, mkt, d, cols, hf_lookback_days=hf_days)
        else:
            df = rr.jeffreys_window(pc, jeff, mkt, d, cols)
        return df["Weight"].reindex(_G["tickers"]).to_numpy()
    from oracle import bayes_oracle as bo
    if kind == 0:
        return bo.conjugate_window(conj, mkt, d, cols, hf_lookback_days=hf_days)["weights"]
    return bo.jeffreys_window(jeff, mkt, d, cols)["weights"]


def _ref_setup(args, mkt, conj, jeff, impl):
    _G.update(mkt=mkt, conj=conj, jeff=jeff, cols=np.arange(args.n_assets), hf_days=args.hf_days, impl=impl,
              tickers=[mkt.tickers[c] for c in range(args.n_assets)])
    if impl == "reference":
        from oracle.ref_import import load_reference, set_universe
        _G["pc"] = load_reference(check=False)
        set_universe(mkt.tickers)


def reference_impl():
    from oracle.ref_import import reference_available
    return "reference" if reference_available() else "port"


def sample_jobs(d_idx, n_windows):
    n = max(1, n_windows // 2)
    sel = np.linspace(0, len(d_idx) - 1, n).round().astype(int)
    sel = np.unique(sel)
    return sel, [(0, int(d_idx[i])) for i in sel] + [(1, int(d_idx[i])) for i in sel]


def host_procs():
    try:
        cores = len(os.sched_getaffinity(0))
    except Exception:
        cores = os.cpu_count() or 1
    return max(1, min(cores, 64))


def blas_threads():
    try:
        from threadpoolctl import threadpool_info
        return int(max([p.get("num_threads", 1) for p in threadpool_info()] or [1]))
    except Exception:
        return 1


def timed_pool(jobs, procs, repeats=1, warm=0):
    """jobs through a fork pool of `procs` single-BLAS-thread workers; returns (seconds per pass, results of the last)."""
    import multiprocessing as mp
    try:
        from threadpoolctl import threadpool_limits
    except Exception:
        threadpool_limits = None
    ctx = mp.get_context("fork")
    lim = threadpool_limits(1) if threadpool_limits else None        # one BLAS thread per worker: windows are independent
    try:
        with ctx.Pool(procs) as pool:
            for _ in range(warm):
                pool.map(_ref_window, jobs, chunksize=1)
            t0 = time.perf_counter()
            for _ in range(repeats):
                res = pool.map(_ref_window, jobs, chunksize=1)
            dt = (time.perf_counter() - t0) / repeats
    finally:
        if lim is not None:
            lim.restore_original_limits()
    return dt, res


def reference_levels(args, mkt, conj, jeff, d_idx, l0_windows=32, l1_dates=3):
    """BASELINE.md section 3 beside the headline CPU figure: L0 (weight-function level, ONE process, NumPy's default
    BLAS threads, CHECK=False), L1 (``backtest_portfolio`` as shipped, CHECK=True, full market_data; the reference's
    own 1-day intraday look-back) and the NumPy port at L0.  Bounded samples; the reference must be importable."""
    from oracle import bayes_oracle as bo
    from oracle import ref_runner as rr
    out = {}
    sel, jobs = sample_jobs(d_idx, l0_windows)
    _ref_setup(args, mkt, conj, jeff, "reference")
    t0 = time.perf_counter()
    for j in jobs:
        _ref_window(j)
    out["L0"] = {"windows_per_s": len(jobs) / (time.perf_counter() - t0), "windows": len(jobs), "processes": 1,
                 "blas_threads": blas_threads(), "what": "calculate_conjugate_hf_mcm_portfolio / calculate_jeffreys_portfolio "
                 "of the unmodified reference on minimal frames, CHECK=False"}
    _G["impl"] = "port"
    t0 = time.perf_counter()
    for j in jobs:
        _ref_window(j)
    out["port_L0"] = {"windows_per_s": len(jobs) / (time.perf_counter() - t0), "windows": len(jobs), "processes": 1,
                      "blas_threads": blas_threads(), "what": "oracle/bayes_oracle.py (NumPy restatement)"}
    _G["impl"] = "reference"
    if l1_dates > 0:
        dd = d_idx[len(d_idx) // 2: len(d_idx) // 2 + l1_dates]
        sec, reb = rr.loop_level(mkt, conj, dd, check=True)
        out["L1"] = {"windows_per_s": reb / sec, "windows": int(reb), "processes": 1, "blas_threads": blas_threads(),
                     "what": "backtest_portfolio as shipped (CHECK=True, universe selection, loop body, 1-day intraday "
                             "look-back) over consecutive rebalance dates, conjugate strategy"}
    return out


def run_reference(args):
    """CPU arm: the unmodified reference (L0-mp) on every host core, a bounded sample of the same windows per step."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    mkt, conj, jeff, d_idx = make_workload(args, 0)
    procs = host_procs()
    impl = reference_impl()
    per_step = max(2 * procs, args.ref_sample)
    sel, jobs = sample_jobs(d_idx, per_step)
    _ref_setup(args, mkt, conj, jeff, impl)
    dt, _ = timed_pool(jobs, procs, repeats=args.steps, warm=args.warmup)
    value = len(jobs) / dt
    sample = (f"{len(jobs)} windows per step ({len(jobs)//2} conjugate + {len(jobs)//2} Jeffreys, stratified over the "
              f"{args.windows} rebalance dates), {procs} worker processes x 1 BLAS thread (level L0-mp)")
    cpu = {"value": value, "unit": UNIT, "cores": procs, "kind": impl, "sample": sample}
    if impl == "reference" and not args.no_levels:
        cpu["levels"] = reference_levels(args, mkt, conj, jeff, d_idx)
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt * 1e3, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": dict(config_dict(args, 1, conj, jeff, args.hf_days), **intraday_config(mkt, conj, d_idx, args.hf_days)),
        "cpu_baseline": cpu,
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
        "note": ("the UNMODIFIED reference (baseline/_ref/src/portfolio_calculations.py: calculate_conjugate_hf_mcm_portfolio "
                 ":819-836 with the 7-day look-back through its own calculate_conjugate_prior_S, calculate_jeffreys_portfolio "
                 ":838-849), CHECK=False, minimal pre-sliced frames (SURVEY 8(c)), NumPy/pandas of this image")
                if impl == "reference" else
                "baseline/_ref/src not staged: fell back to oracle/bayes_oracle.py (NumPy restatement pinned by tests/golden)",
    }
    print(json.dumps(line), flush=True)


# ----------------------------------------------------------------------------- our arm
class _StdoutToStderr:
    """NCCL prints its version banner on STDOUT when the communicator is created; the contract is ONE JSON line on
    stdout, so file descriptor 1 points at stderr while the process group comes up."""

    def __enter__(self):
        sys.stdout.flush()
        self.saved = os.dup(1)
        os.dup2(2, 1)
        return self

    def __exit__(self, *exc):
        sys.stdout.flush()
        os.dup2(self.saved, 1)
        os.close(self.saved)
        return False


def measure_dgemm_peak(torch, dev):
    n = 8192
    a = torch.randn(n, n, dtype=torch.float64, device=dev)
    b = torch.randn(n, n, dtype=torch.float64, device=dev)
    best = 1e30
    for i in range(6):
        e0 = torch.cuda.Event(enable_timing=True)
        e1 = torch.cuda.Event(enable_timing=True)
        e0.record()
        c = a @ b
        e1.record()
        torch.cuda.synchronize()
        if i:
            best = min(best, e0.elapsed_time(e1))
    del a, b, c
    torch.cuda.empty_cache()
    return 2.0 * n ** 3 / (best * 1e-3) / 1e12


def run_ours(args):
    import torch
    import torch.distributed as dist
    from incorporating_different_sources_b200.engine import BayesEngine, upload_synthetic
    from incorporating_different_sources_b200.windows import ffill_rows, plan_daily_windows, trim_intraday

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the CUDA path has no CPU fallback (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        with _StdoutToStderr():
            dist.init_process_group("nccl", device_id=dev)
            warm = torch.zeros(1, device=dev)
            dist.all_reduce(warm)                  # creates the communicator (and prints the banner) here
            torch.cuda.synchronize()
    n_gpus = world

    peaks = {}
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            peaks = json.load(f)
    except Exception:
        pass
    hbm_peak = float(peaks.get("hbm_gbs", 6650.0))
    hbm_src = "MEASURED_PEAKS.json hbm_gbs" if "hbm_gbs" in peaks else "fallback 6650 GB/s (B200_PROFILING.md)"
    dgemm_tf = measure_dgemm_peak(torch, dev)

    mkt, conj, jeff, d_idx = make_workload(args, rank)
    N, W = args.n_assets, len(d_idx)
    eng = BayesEngine(local)
    # pinned host copies of the inputs (the e2e leg copies them every step)
    def pin(a):
        t = torch.empty(a.shape, dtype=torch.float64).pin_memory()
        v = t.numpy()
        v[...] = a
        return t, v
    keep = []
    host = {}
    cb = plan_daily_windows(conj, mkt.dates, d_idx, mkt.hf_ts, hf_lookback_days=args.hf_days)
    jb = plan_daily_windows(jeff, mkt.dates, d_idx, need_hf=False)
    # the 1,007 days of history before the first rebalance date are read by the DAILY windows only: their intraday
    # bars belong to no window (the reference never touches them either) and are not uploaded
    hf_row_lo, hf_row_hi = trim_intraday(cb)
    hf_used = mkt.hf_prices[hf_row_lo:hf_row_hi]
    for name, arr in (("prices", mkt.prices), ("caps", mkt.caps), ("hf_prices", hf_used),
                      ("mcm", np.stack([mkt.vix, mkt.epu])), ("rf_row", ffill_rows(mkt.dates, mkt.dates, mkt.rf))):
        t, v = pin(arr)
        keep.append(t)
        host[name] = v
    h2d_bytes = int(sum(v.nbytes for v in host.values()))
    m_hf = int((cb.hf_hi - cb.hf_lo - 1).max())

    eng.upload_market(**host)
    out_c = {"weights": torch.empty((W, N), dtype=torch.float64, device=dev),
             "status": torch.empty((W,), dtype=torch.int32, device=dev)}
    out_j = {"weights": torch.empty((W, N), dtype=torch.float64, device=dev),
             "status": torch.empty((W,), dtype=torch.int32, device=dev)}
    gathered_c = gathered_j = None
    if world > 1:
        gathered_c = torch.empty((world, W, N), dtype=torch.float64, device=dev)
        gathered_j = torch.empty((world, W, N), dtype=torch.float64, device=dev)

    def step_device():
        eng.prepare_market()
        eng.conjugate(cb, outputs=("weights", "status"), into=out_c)
        if world > 1:
            # the gather of the conjugate weights travels over NVLink while the Jeffreys windows are computed
            # (NCCL's stream waits for the kernels queued so far; the compute stream goes on)
            hc = dist.all_gather_into_tensor(gathered_c.view(-1), out_c["weights"].view(-1), async_op=True)
        eng.jeffreys(jb, outputs=("weights", "status"), into=out_j)
        if world > 1:
            hj = dist.all_gather_into_tensor(gathered_j.view(-1), out_j["weights"].view(-1), async_op=True)
            hc.wait()
            hj.wait()

    hw_c, hw_cv = pin(np.zeros((W, N)))
    hw_j, hw_jv = pin(np.zeros((W, N)))
    hs_ct = torch.zeros(W, dtype=torch.int32).pin_memory()
    hs_jt = torch.zeros(W, dtype=torch.int32).pin_memory()
    hs_c, hs_j = hs_ct.numpy(), hs_jt.numpy()
    d2h_bytes = int(hw_cv.nbytes + hw_jv.nbytes + hs_c.nbytes + hs_j.nbytes)

    # segments of the pipelined upload: one solver wave of ready windows per segment, then halves (see DESIGN 4.6)
    e2e_fractions = eng.plan_upload_fractions(cb, hf_used.shape[0])

    # long look-backs take the pre-summed day-block path, which is not pipelined against the upload inside one call:
    # the conjugate batch is cut along the upload segments instead, and each sub-batch waits for its own segments only
    from incorporating_different_sources_b200.windows import split_batch_by_fractions
    sub_batches = None
    if args.hf_days >= 12 and e2e_fractions:
        sub_batches = split_batch_by_fractions(cb, e2e_fractions, hf_used.shape[0])

    def step_e2e():
        # pinned host buffers -> HBM (the 1.6 GB intraday block in segments on the copy stream), Jeffreys first
        # because it does not read intraday data and so overlaps the transfer, then conjugate, pipelined against
        # the remaining segments; the calls only queue work (async outputs), so the host plans the conjugate
        # batch while the GPU runs Jeffreys; weights and status flags are in pinned host memory after synchronize()
        eng.set_async_outputs(True)
        eng.set_upload_fractions(e2e_fractions)
        eng.upload_market(**host, async_copy=True)
        eng.jeffreys(jb, outputs=("weights", "status"), into={"weights": hw_jv, "status": hs_j})
        if sub_batches:
            for i0, i1, sb in sub_batches:
                eng.conjugate(sb, outputs=("weights", "status"), into={"weights": hw_cv[i0:i1], "status": hs_c[i0:i1]})
        else:
            eng.conjugate(cb, outputs=("weights", "status"), into={"weights": hw_cv, "status": hs_c})
        eng.synchronize()
        eng.set_async_outputs(False)
        eng.set_upload_fractions(None)

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    def max_over_ranks(x):
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    # ---- device-resident timing
    for _ in range(args.warmup):
        step_device()
    barrier()
    eng.set_stage_timing(True)
    eng.stage_times()
    eng.gram_work()
    eng.solve_work()
    launches0 = eng.launch_count
    sampler = ClockSampler(local)
    sampler.start()
    e0 = torch.cuda.Event(enable_timing=True)
    e1 = torch.cuda.Event(enable_timing=True)
    barrier()
    e0.record()
    for _ in range(args.steps):
        step_device()
    e1.record()
    barrier()
    clocks = sampler.stop()
    ms = max_over_ranks(e0.elapsed_time(e1) / args.steps)
    stages = eng.stage_times()
    gwork = eng.gram_work()
    swork = eng.solve_work()
    eng.set_stage_timing(False)
    launches = (eng.launch_count - launches0) // args.steps + (2 if world > 1 else 0)      # + the two all-gathers
    status_bad = int((out_c["status"] != 0).sum().item() + (out_j["status"] != 0).sum().item())
    value = n_gpus * 2 * W / (ms * 1e-3)
    if args.dump_outputs and rank == 0:
        # what a caller of the timed path receives from its last step: the (all-gathered) weights and the status flags
        wc, wj = (out_c["weights"], out_j["weights"]) if world == 1 else (gathered_c.view(-1, N), gathered_j.view(-1, N))
        dump_outputs(args.dump_outputs, {"conjugate_weights": wc.cpu().numpy(), "jeffreys_weights": wj.cpu().numpy(),
                                         "conjugate_status": out_c["status"].cpu().numpy(),
                                         "jeffreys_status": out_j["status"].cpu().numpy()})

    # ---- end-to-end timing through the host-buffer API
    step_e2e()
    barrier()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        step_e2e()
    torch.cuda.synchronize()
    e2e_s = max_over_ranks((time.perf_counter() - t0) / args.steps)
    e2e_value = n_gpus * 2 * W / e2e_s
    if sub_batches:      # sub-batches anchor their block grids differently: same sums, different association
        ref_w = out_c["weights"].cpu().numpy()
        e2e_match = bool(np.max(np.abs(hw_cv - ref_w)) <= 1e-10 * np.max(np.abs(ref_w)))
    else:
        e2e_match = bool(np.array_equal(hw_cv, out_c["weights"].cpu().numpy()))
    # platform limit of the e2e leg: every rank copies a buffer of its intraday block's size at once (plain cudaMemcpyAsync)
    hf_t = keep[2]
    torch.cuda.synchronize()
    dst = torch.empty(hf_t.shape, dtype=torch.float64, device=dev)
    dst.copy_(hf_t, non_blocking=True)
    barrier()
    t0 = time.perf_counter()
    for _ in range(3):
        dst.copy_(hf_t, non_blocking=True)
    torch.cuda.synchronize()
    h2d_s = max_over_ranks((time.perf_counter() - t0) / 3)
    del dst
    h2d_ceiling = {"bytes_per_rank": int(hf_t.numel() * 8), "ranks": world, "ms": h2d_s * 1e3,
                   "per_rank_gbs": hf_t.numel() * 8 / h2d_s / 1e9, "aggregate_gbs": world * hf_t.numel() * 8 / h2d_s / 1e9,
                   "what": "pinned -> device cudaMemcpyAsync of the intraday block alone, all ranks at once, max over ranks"}

    if rank == 0:
        work = algorithmic_work(N, W, conj["rolling_window"], m_hf, jeff["rolling_window"])
        k = args.steps
        g_ms = stages["gram"]["ms"] / k
        s_ms = stages["solve"]["ms"] / k
        p_ms = stages["prep"]["ms"] / k
        l_ms = stages["logret"]["ms"] / k
        nt = (N + 127) // 128
        npairs = nt * (nt + 1) // 2
        tile = 128 * 128
        gram_conv_tf = work["gram_flops"] / (g_ms * 1e-3) / 1e12 if g_ms > 0 else 0.0
        gram_exec_flops = 2.0 * npairs * tile * (gwork["k_rows"] + gwork["precompute_rows"]) / k
        gram_add_bytes = gwork["add_blocks"] * npairs * tile * 8.0 / k
        gram_scratch_flops = 2.0 * npairs * tile * gwork["full_rows"] / k
        c_ms = stages["chain"]["ms"] / k
        chol_flops = N ** 3 / 3.0 + 4.0 * N * N
        factored, chained = swork["factored"] / k, swork["chained"] / k
        # the kernel's own work: only the windows it factorises (Jeffreys windows of consecutive dates are solved
        # relative to every 8th window by jeffreys_chain_kernel and are NOT charged to the Cholesky kernel)
        solve_tf = factored * chol_flops / (s_ms * 1e-3) / 1e12 if s_ms > 0 else 0.0
        groups = factored - W if chained > 0 else 0.0           # Jeffreys base windows = groups of the chain kernel
        chain_flops = groups * (64.0 * N * N + 2048.0 * N)       # 32 right-hand sides forward + backward, Z'Z
        prof = {}
        try:
            with open(os.path.join(ROOT, "profiles", "kernel_traffic.json")) as f:
                prof = json.load(f)
        except Exception:
            pass
        # the traffic figures come from an ncu launch list (tools/kernel_traffic.py); say whether it was taken on the
        # kernel sources this run was built from
        try:
            sys.path.insert(0, os.path.join(ROOT, "tools"))
            from sass_summary import csrc_sha16
            tree_sha = csrc_sha16()
        except Exception:
            tree_sha = None
        traffic_source = {"file": "profiles/kernel_traffic.json", "profiled_csrc_sha16": prof.get("csrc_sha16"),
                          "this_tree_csrc_sha16": tree_sha,
                          "same_kernel_sources": bool(tree_sha and prof.get("csrc_sha16") == tree_sha),
                          "how": "ncu --metrics dram__bytes_read.sum,dram__bytes_write.sum launch list of this command, median per launch"}
        gram_exec_tf = gram_exec_flops / (g_ms * 1e-3) / 1e12 if g_ms > 0 else 0.0
        gram_roof = {
            "kernel": "gram_dmma_kernel (per step: block precompute + conjugate S1 + Jeffreys J launches) + run / scan kernels",
            "bound": "tensor", "achieved": gram_exec_tf, "peak": dgemm_tf, "unit": "TFLOP/s",
            "frac": gram_exec_tf / dgemm_tf if dgemm_tf > 0 else None,
            "traffic": prof.get("gram_dram_bytes_per_launch"), "traffic_source": traffic_source,
            "ms_per_step": g_ms, "share_of_step": g_ms / ms if ms > 0 else None,
            "flops_convention": "EXECUTED DMMA work: 2 * 128 * 128 flops per contracted k-row and lower-triangular tile pair (window "
                                "launches + block precompute); the stage also streams precomputed block tiles from L2 "
                                "(block_tiles_added_gbs), which bounds the conjugate main launch",
            "conventional_tflops": gram_conv_tf,
            "conventional_note": "SURVEY 8(d) convention (full-matrix 2*N^2*K per window, every window contracted from scratch): "
                                 "NOT a utilisation -- overlapping windows share block Gram tiles, so only "
                                 "executed_share_of_from_scratch of those flops are issued",
            "executed_share_of_from_scratch": gram_exec_flops / gram_scratch_flops if gram_scratch_flops > 0 else None,
            "block_tiles_added_gbs": gram_add_bytes / (g_ms * 1e-3) / 1e9 if g_ms > 0 else None,
        }
        solve_roof = {
            "kernel": "chol_solve_kernel (2 launches per step: every conjugate window, every 8th Jeffreys window)",
            "windows_factorised_per_step": factored, "windows_solved_relative_to_a_base_per_step": chained,
            "bytes_per_launch_convention": "8N^2 + 16N per factorised window",
            "bound": "tensor", "achieved": solve_tf, "peak": dgemm_tf, "unit": "TFLOP/s",
            "frac": solve_tf / dgemm_tf if dgemm_tf > 0 else None,
            "traffic": prof.get("solve_dram_bytes_per_launch"), "traffic_source": traffic_source,
            "algorithmic_bytes_per_launch": W * (8.0 * N * N + 16.0 * N),
            "ms_per_step": s_ms, "share_of_step": s_ms / ms if ms > 0 else None,
            "flops_convention": "SURVEY 8(d): N^3/3 + 4N^2 per FACTORISED window (Cholesky + two triangular solves + v1)",
            "solve_stage_conventional_tflops": work["solve_flops"] / ((s_ms + c_ms) * 1e-3) / 1e12 if s_ms + c_ms > 0 else None,
            "solve_stage_note": "conventional = every one of the 2W windows charged a full factorisation, over the time of "
                                "chol_solve_kernel + jeffreys_chain_kernel; not a utilisation figure",
            "achieved_gbs_vs_hbm": factored * (8.0 * N * N + 16.0 * N) / (s_ms * 1e-3) / 1e9 if s_ms > 0 else None,
            "hbm_peak_gbs": hbm_peak,
        }
        dominant = solve_roof if s_ms >= g_ms else gram_roof
        other = gram_roof if dominant is solve_roof else solve_roof
        dominant = dict(dominant, peak_source="cuBLAS DGEMM 8192^3 (torch.matmul f64) measured live in this run; "
                                              "MEASURED_PEAKS.json has no FP64 figure")
        logret_bytes = 8.0 * (mkt.prices.shape[0] + hf_used.shape[0]) * (N + eng_ld(N))
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": n_gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": dict(config_dict(args, n_gpus, conj, jeff, args.hf_days),
                           **intraday_config(mkt, conj, d_idx, args.hf_days)),
            "clocks": clocks,
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d_bytes, "d2h_bytes_per_step": d2h_bytes,
                    "ms_per_step": e2e_s * 1e3, "matches_device_path": e2e_match, "steps": args.steps,
                    "inputs": "host buffers pinned once outside the timed region; windows planned once outside it",
                    "conjugate_sub_batches": len(sub_batches) if sub_batches else 1,
                    "h2d_ceiling": h2d_ceiling,
                    "h2d_ms_at_ceiling": h2d_bytes / (h2d_ceiling["per_rank_gbs"] * 1e9) * 1e3,
                    "frac_of_h2d_ceiling": (h2d_bytes / (h2d_ceiling["per_rank_gbs"] * 1e9)) / e2e_s},
            "gpu_launches": int(launches),
            "roofline": dominant,
            "stages": {
                "second_kernel": other,
                "logret": {"ms": l_ms, "bound": "hbm", "achieved_gbs": logret_bytes / (l_ms * 1e-3) / 1e9 if l_ms > 0 else None,
                           "peak_gbs": hbm_peak, "peak_source": hbm_src},
                "prep": {"ms": p_ms, "bound": "hbm", "achieved_gbs": work["prep_bytes"] / (p_ms * 1e-3) / 1e9 if p_ms > 0 else None,
                         "peak_gbs": hbm_peak, "note": "algorithmic bytes: each window charged its own rows; served mostly from L2"},
                "gram": {"ms": g_ms}, "solve": {"ms": s_ms},
                "chain": {"ms": c_ms, "kernel": "jeffreys_chain_kernel (one CTA per group of 8 consecutive Jeffreys windows)",
                          "windows": chained, "groups": groups, "bound": "fp64 pipe (plain DFMA) + latency",
                          "achieved_tflops": chain_flops / (c_ms * 1e-3) / 1e12 if c_ms > 0 else None,
                          "flops_convention": "64 N^2 + 2048 N per group: 32 right-hand sides through L and L', and Z'Z"},
            },
            "windows_flagged_singular": status_bad,
        }
        # SURVEY 8(d): lower bound of the WHOLE step for a reuse-exploiting implementation, so that the per-stage
        # figures above cannot be read as > 100 %: every distinct return row enters one symmetric rank-1 update per
        # phase (N(N+1) flops), every window needs its own factorisation and solves; every input element is read once
        # and every weight written once.
        rows_unique = (mkt.prices.shape[0] - 1) * 2 + (hf_used.shape[0] - 1)      # daily rows serve both priors
        lb_flops = rows_unique * float(N) * (N + 1) + work["solve_flops"]
        lb_bytes = 8.0 * N * (2 * mkt.prices.shape[0] + hf_used.shape[0]) + 8.0 * N * 2 * W
        lb_ms = max(lb_flops / (dgemm_tf * 1e12), lb_bytes / (hbm_peak * 1e9)) * 1e3
        line["step_lower_bound"] = {
            "unique_flops": lb_flops, "unique_bytes": lb_bytes,
            "ms_at_peak": lb_ms, "bound": "tensor" if lb_flops / (dgemm_tf * 1e12) > lb_bytes / (hbm_peak * 1e9) else "hbm",
            "achieved_frac": lb_ms / ms if ms > 0 else None,
            "note": "unique work of the backtest (each return row contracted once per phase, one Cholesky + solves per "
                    "window, inputs read once) at the measured DGEMM / HBM peaks, over the measured step"}
        if n_gpus == 1 and not args.no_cpu:
            line["cpu_baseline"], line["parity_max_rel_err"], line["parity"] = cpu_baseline(args, mkt, conj, jeff, d_idx, out_c, out_j)
        if n_gpus == 1 and not args.no_widened:
            line["widened"] = widened_estimators(args, torch, eng, mkt, jeff, d_idx, dgemm_tf, not args.no_cpu)
        if n_gpus == 1 and not args.no_loop:
            line["loop_e2e"] = loop_level(args, eng, mkt, conj, jeff, d_idx)
        print(json.dumps(line), flush=True)
    eng.close()
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def loop_level(args, eng, mkt, conj, jeff, d_idx):
    """SURVEY 8(f) ranks 1-2, OUTSIDE the timed region of the headline metric: the reference's loop-level entry point
    ``backtest_portfolio(portfolio_spec, ts_start_date, ts_end_date, market_data)`` (:1221-1238) on pandas frames, whole
    backtest, wall clock: calendar, universe selection for every date (vectorised, :611-658), ONE upload of the market
    into the resident pool, device gathers per asset set, batched weights, loop-body kernel, pandas containers out.
    The reference's own loop (level L1 of the CPU arm) is the figure to set beside it."""
    import pandas as pd
    from incorporating_different_sources_b200 import portfolio_calculations as pcg
    md = mkt.market_data()                      # the 10-key dict of data_handling.py:282-291 (input boundary, not timed)
    start, end = pd.Timestamp(mkt.dates[d_idx[0]]), pd.Timestamp(mkt.dates[d_idx[-1]])
    out = {"entry_point": "backtest_portfolio(spec, start, end, market_data) with pandas frames, wall clock, everything inside",
           "n_assets": args.n_assets, "rebalance_dates": int(len(d_idx))}
    for name, spec, kw in (("jeffreys", jeff, {}), ("conjugate", conj, {"hf_lookback_days": args.hf_days})):
        best = None
        for _ in range(2):                      # second pass: allocations of the first one are reused
            tm = {}
            t0 = time.perf_counter()
            res = pcg.backtest_portfolio(spec, start, end, md, engine=eng, timings=tm, **kw)
            dt = time.perf_counter() - t0
            if best is None or dt < best["seconds"]:
                r = res["portfolio_simple_returns_series"].to_numpy()
                best = dict(seconds=dt, windows_per_s=len(d_idx) / dt, phases_s={k: v for k, v in tm.items() if k.endswith("_s")},
                            asset_sets=tm.get("asset_sets"), returns=int(len(r)), returns_finite=bool(np.isfinite(r).all()),
                            turnover_rows=int(len(res["portfolio_turnover_series"])),
                            metrics_shape=list(res["portfolio_weights_metrics_df"].shape))
        out[name] = best
    # the experiment the reference ships (portfolio_specs.py:54-62): top 50 by cap, MONTHLY rebalancing, 250-WEEK window,
    # weekly 7-day intraday look-back -- windows that are neither daily nor consecutive (no block reuse between them) and
    # a universe that changes from month to month (one device gather + one batched call per distinct asset set)
    ship = dict(weighting_strategy="conjugate_hf_vix_vw", size=50, risk_aversion=5, turnover_cost=15,
                rebalancing_frequency="monthly", rolling_window=250, rolling_window_frequency="weekly", mcm_scaling=1,
                display_name="Conjugate HF-VIX VW (shipped spec)")
    first = max(int(d_idx[0]), 1300)             # 250 complete weeks of history before the first rebalance
    if first < int(d_idx[-1]) - 60:
        tm = {}
        t0 = time.perf_counter()
        res = pcg.backtest_portfolio(ship, pd.Timestamp(mkt.dates[first]), end, md, engine=eng, timings=tm)
        dt = time.perf_counter() - t0
        r = res["portfolio_simple_returns_series"].to_numpy()
        out["shipped_spec"] = dict(spec="N=50 of 500, monthly rebalancing, 250-week window, gamma 5, 15 bp", seconds=dt,
                                   rebalances=tm.get("rebalances"), asset_sets=tm.get("asset_sets"),
                                   rebalances_per_s=tm.get("rebalances", 0) / dt, trading_days=int(len(r)),
                                   phases_s={k: v for k, v in tm.items() if k.endswith("_s")},
                                   returns_finite=bool(np.isfinite(r).all()))
    return out


def eng_ld(N):
    return (N + 15) // 16 * 16


def cpu_baseline(args, mkt, conj, jeff, d_idx, out_c, out_j):
    """The reference's own CPU path (unmodified sources, level L0-mp: every host core, one BLAS thread per worker)
    over a bounded, stratified sample of the step's windows; doubles as a parity check of the GPU weights against
    the unmodified reference AND against the NumPy port.  Falls back to the port alone when baseline/_ref/src is
    not staged."""
    procs = host_procs()
    impl = reference_impl()
    wc = out_c["weights"].cpu().numpy()
    wj = out_j["weights"].cpu().numpy()

    def worst_err(sel, res):
        n = len(sel)
        worst = 0.0
        for k, i in enumerate(sel):
            for got, ref in ((wc[i], res[k]), (wj[i], res[n + k])):
                worst = max(worst, float(np.max(np.abs(got - ref)) / np.max(np.abs(ref))))
        return worst

    parity = {}
    sel, jobs = sample_jobs(d_idx, args.cpu_sample)
    _ref_setup(args, mkt, conj, jeff, "port")
    dt_port, res = timed_pool(jobs, procs)
    parity["vs_port"] = worst_err(sel, res)
    port = {"value": len(jobs) / dt_port, "unit": UNIT, "cores": procs, "kind": "port",
            "sample": f"{len(jobs)} windows, oracle/bayes_oracle.py, {procs} worker processes x 1 BLAS thread"}
    if impl != "reference":
        return port, parity["vs_port"], parity
    sel, jobs = sample_jobs(d_idx, args.cpu_sample)
    _ref_setup(args, mkt, conj, jeff, "reference")
    dt, res = timed_pool(jobs, procs)
    parity["vs_reference"] = worst_err(sel, res)
    cpu = {"value": len(jobs) / dt, "unit": UNIT, "cores": procs, "kind": "reference",
           "sample": f"{len(jobs)} windows ({len(jobs)//2} conjugate + {len(jobs)//2} Jeffreys, stratified over the "
                     f"{len(d_idx)} rebalance dates), the unmodified reference (baseline/_ref/src) at level L0-mp: "
                     f"{procs} worker processes x 1 BLAS thread",
           "port": port}
    if not args.no_levels:
        cpu["levels"] = reference_levels(args, mkt, conj, jeff, d_idx)
    return cpu, max(parity.values()), parity


def widened_estimators(args, torch, eng, mkt, jeff, d_idx, dgemm_tf, with_cpu):
    """SURVEY 8(f) rank 3, measured OUTSIDE the timed region of the headline metric: Jorion (:851-895) and the
    Ledoit-Wolf shrinkage closed form (:703-758) over the same 4,150 rebalance dates (rolling_window of the Jeffreys
    leg), device resident, CUDA events; a few windows re-checked against the oracle and timed on the CPU."""
    from incorporating_different_sources_b200.windows import plan_daily_windows
    from oracle import bayes_oracle as bo
    N, W = args.n_assets, len(d_idx)
    dev = torch.device("cuda", eng.device)
    out = {"weights": torch.empty((W, N), dtype=torch.float64, device=dev),
           "status": torch.empty((W,), dtype=torch.int32, device=dev)}
    res = {}
    cols = np.arange(N)
    sel = np.linspace(0, W - 1, 6).round().astype(int)
    for name, run, oracle in (("jorion", eng.jorion, bo.jorion_window), ("shrinkage", eng.shrinkage, bo.shrinkage_window)):
        spec = dict(jeff, weighting_strategy=name, display_name=name)
        batch = plan_daily_windows(spec, mkt.dates, d_idx, need_hf=False)
        run(batch, outputs=("weights", "status"), into=out)
        torch.cuda.synchronize()
        eng.set_stage_timing(True)
        eng.stage_times()
        eng.solve_work()
        l0 = eng.launch_count
        e0 = torch.cuda.Event(enable_timing=True)
        e1 = torch.cuda.Event(enable_timing=True)
        reps = 3
        e0.record()
        for _ in range(reps):
            run(batch, outputs=("weights", "status"), into=out)
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / reps
        st = eng.stage_times()
        sw = eng.solve_work()
        eng.set_stage_timing(False)
        chol = N ** 3 / 3.0 + (6.0 if name == "jorion" else 4.0) * N * N
        s_ms = st["solve"]["ms"] / reps
        fact = sw["factored"] / reps
        r = {"windows_per_s": W / (ms * 1e-3), "ms_per_batch": ms, "windows": W, "rolling_window": jeff["rolling_window"],
             "gpu_launches": int((eng.launch_count - l0) // reps),
             "stages_ms": {k: st[k]["ms"] / reps for k in ("prep", "gram", "solve", "chain")},
             "windows_factorised": fact, "windows_solved_relative_to_a_base": sw["chained"] / reps,
             "solve_tflops": fact * chol / (s_ms * 1e-3) / 1e12 if s_ms > 0 else None,
             "solve_frac_of_dgemm_peak": fact * chol / (s_ms * 1e-3) / 1e12 / dgemm_tf if s_ms > 0 and dgemm_tf > 0 else None,
             "windows_flagged_singular": int((out["status"] != 0).sum().item())}
        if with_cpu:
            w = out["weights"].cpu().numpy()
            worst = 0.0
            t0 = time.perf_counter()
            for i in sel:
                ref = oracle(spec, mkt, int(d_idx[i]), cols)["weights"]
                worst = max(worst, float(np.max(np.abs(w[i] - ref)) / np.max(np.abs(ref))))
            r["cpu_port_windows_per_s"] = len(sel) / (time.perf_counter() - t0)
            r["parity_max_rel_err"] = worst
        res[name] = r
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--n-assets", type=int, default=500)
    ap.add_argument("--windows", type=int, default=4150)
    ap.add_argument("--hf-days", type=int, default=7)
    ap.add_argument("--cpu-sample", type=int, default=1024, help="windows of the in-run CPU baseline / parity check (~10 s)")
    ap.add_argument("--ref-sample", type=int, default=1024, help="windows per step of the --impl reference arm (~2 s per step)")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-levels", action="store_true", help="skip the L0 / L1 / port side measurements of the CPU arm")
    ap.add_argument("--no-loop", action="store_true", help="skip the loop-level (backtest_portfolio) measurement (SURVEY 8(f))")
    ap.add_argument("--no-widened", action="store_true", help="skip the Jorion / shrinkage measurements (SURVEY 8(f))")
    ap.add_argument("--config", default="C2", choices=["C1", "C2", "C3", "C4", "C5"],
                    help="BASELINE.json configuration (default C2 = the headline metric); see bench_configs.py")
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"],
                    help="N > 1: weak = one independent path per GPU; strong = ONE backtest split by date range (north star)")
    ap.add_argument("--paths", type=int, default=64, help="C5: independent synthetic paths in total")
    ap.add_argument("--path-pool", type=int, default=2, help="C5: distinct generated markets per GPU the paths cycle through")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="C2: write the weights and status flags of the last timed step as DIR/<name>.npy (float64)")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be >= 1 and --warmup >= 0")
    if args.dump_outputs and (args.impl != "ours" or args.config != "C2" or args.scaling != "weak"):
        ap.error("--dump-outputs applies to the C2 workload of --impl ours with --scaling weak")
    if args.impl == "reference":
        run_reference(args)
    elif args.config != "C2" or args.scaling == "strong":
        import bench_configs
        bench_configs.dispatch(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
