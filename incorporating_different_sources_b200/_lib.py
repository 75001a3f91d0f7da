"""ctypes binding of ``libbayes_portfolio.so`` (see ``include/bayes_portfolio.h``).

The library is the product: there is no CPU fallback.  Loading works without a GPU (so that the
CPU test-suite can check the exported symbols), but ``bp_init`` fails loudly when no sm_100 device
is present, and every engine call raises if the library is missing.
"""
from __future__ import annotations

import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "libbayes_portfolio.so")

BP_NSCAL = 12
EST_JORION, EST_SHRINKAGE = 1, 2
SCAL_JORION = dict(mu_g=0, lambda_hat=1, v_hat=2, q=4, one_vinv_one=5)
SCAL_LW = dict(shrinkage=0, mu=1, beta=2, delta=4)
SCAL = dict(n0=0, n1=1, alpha=2, beta=3, c=4, v0=5, m=6, sum_a=7, v1=8, mcm_avg=9, anorm1=10, rcond=11)

BP_OK, BP_ERR_INVALID, BP_ERR_CUDA, BP_ERR_NO_DEVICE, BP_ERR_STATE = 0, 1, 2, 3, 4

EXPORTED = [
    "bp_last_error", "bp_version", "bp_init", "bp_destroy", "bp_set_stream", "bp_synchronize",
    "bp_set_workspace_limit", "bp_device_info", "bp_launch_count", "bp_upload_market",
    "bp_prepare_market", "bp_stats_batched", "bp_hf_cov_batched", "bp_conjugate_batched",
    "bp_jeffreys_batched", "bp_set_stage_timing", "bp_get_stage_times",
    "bp_excess_returns", "bp_quadratic_form", "bp_dense_posterior", "bp_moments_batched",
    "bp_upload_market_async", "bp_backtest_batched", "bp_get_gram_work", "bp_set_reuse_min_windows", "bp_set_upload_pipeline", "bp_set_async_outputs",
    "bp_set_resampled", "bp_estimator_batched", "bp_set_jeffreys_chain", "bp_get_solve_work",
    "bp_set_upload_fractions", "bp_solve_wave_windows", "bp_set_hf_presum_min_days", "bp_wait_upload", "bp_upload_pool", "bp_select_market", "bp_path_metrics",
    "bp_select_windows",
    "bp_solve_batched", "bp_set_condition_estimate",
]
BP_NSTAGE = 8
STAGES = ("logret", "prep", "gram", "solve", "chain", "cond")

c_double_p = C.POINTER(C.c_double)
c_int_p = C.POINTER(C.c_int)


class MarketDesc(C.Structure):
    _fields_ = [
        ("n_assets", C.c_int), ("n_days", C.c_int), ("n_hf_rows", C.c_longlong),
        ("prices", C.c_void_p), ("caps", C.c_void_p), ("hf_prices", C.c_void_p),
        ("mcm", C.c_void_p), ("n_mcm", C.c_int), ("rf_row", C.c_void_p),
    ]


class WindowBatchDesc(C.Structure):
    _fields_ = [
        ("n_windows", C.c_int), ("rolling_window", C.c_int),
        ("day_row", C.c_void_p), ("span_days", C.c_void_p), ("hf_lo", C.c_void_p), ("hf_hi", C.c_void_p),
        ("mcm_index", C.c_int), ("mcm_scaling", C.c_double), ("risk_aversion", C.c_double),
        ("prior_weights", C.c_int), ("mcm_rows", C.c_int), ("prior_n", C.c_void_p),
        ("resampled", C.c_int), ("extra_row", C.c_void_p), ("caps_row", C.c_void_p),
    ]


class ResampledDesc(C.Structure):
    _fields_ = [("n_rows", C.c_int), ("num_row", C.c_void_p), ("den_row", C.c_void_p), ("rf_row", C.c_void_p),
                ("mcm", C.c_void_p)]


class Outputs(C.Structure):
    _fields_ = [(k, C.c_void_p) for k in
                ("weights", "nu", "w1", "t", "w0", "rhs", "scalars", "status", "T", "S0", "S1")]


class DenseProblem(C.Structure):
    _fields_ = [
        ("n_assets", C.c_int), ("jeffreys", C.c_int), ("rolling_window", C.c_int), ("risk_aversion", C.c_double),
        ("T", C.c_void_p), ("t", C.c_void_p), ("S0", C.c_void_p), ("w0", C.c_void_p), ("n0", C.c_double),
        ("n1", C.c_void_p), ("c", C.c_void_p), ("S1", C.c_void_p), ("w1", C.c_void_p),
    ]


class DenseResult(C.Structure):
    _fields_ = [(k, C.c_void_p) for k in ("scalars", "S1", "w1", "nu", "weights", "status")]


class SolveDesc(C.Structure):
    _fields_ = [
        ("n_windows", C.c_int), ("n_assets", C.c_int), ("jeffreys", C.c_int), ("estimator", C.c_int),
        ("n_returns", C.c_int), ("risk_aversion", C.c_double), ("S", C.c_void_p), ("rhs", C.c_void_p),
        ("n1", C.c_void_p),
    ]


class BacktestDesc(C.Structure):
    _fields_ = [
        ("n_rebalances", C.c_int), ("reb_row", C.c_void_p), ("last_row", C.c_int), ("weights", C.c_void_p),
        ("member", C.c_void_p),
        ("distance_scale", C.c_double), ("turnover_cost_bps", C.c_double),
        ("returns", C.c_void_p), ("turnover", C.c_void_p), ("metrics", C.c_void_p),
    ]


class LibraryMissing(RuntimeError):
    pass


_lib = None


class PoolSelect(C.Structure):
    _fields_ = [("n_cols", C.c_int), ("cols", C.c_void_p), ("day_lo", C.c_int), ("day_hi", C.c_int),
                ("hf_lo", C.c_longlong), ("hf_hi", C.c_longlong)]


class WindowSelect(C.Structure):
    _fields_ = [("n_windows", C.c_int), ("n_cols", C.c_int), ("cols", C.c_void_p), ("day_lo", C.c_void_p),
                ("day_hi", C.c_void_p), ("day_off", C.c_void_p), ("hf_lo", C.c_void_p), ("hf_hi", C.c_void_p),
                ("hf_off", C.c_void_p)]


def load():
    """Load the shared library (building is the job of ``__graft_entry__.build()``)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise LibraryMissing(
            f"{LIB_PATH} is missing: build it with `python -m incorporating_different_sources_b200.build` "
            "(there is no CPU fallback for the CUDA path)")
    lib = C.CDLL(LIB_PATH)
    lib.bp_last_error.restype = C.c_char_p
    lib.bp_version.restype = C.c_int
    lib.bp_init.argtypes = [C.c_int, C.POINTER(C.c_void_p)]
    lib.bp_destroy.argtypes = [C.c_void_p]
    lib.bp_set_stream.argtypes = [C.c_void_p, C.c_void_p]
    lib.bp_synchronize.argtypes = [C.c_void_p]
    lib.bp_wait_upload.argtypes = [C.c_void_p]
    lib.bp_upload_pool.argtypes = [C.c_void_p, C.POINTER(MarketDesc)]
    lib.bp_select_market.argtypes = [C.c_void_p, C.POINTER(PoolSelect)]
    lib.bp_select_windows.argtypes = [C.c_void_p, C.POINTER(WindowSelect)]
    lib.bp_path_metrics.argtypes = [C.c_void_p, C.c_int, C.c_int, c_double_p, c_double_p, C.c_double, c_double_p]
    lib.bp_set_workspace_limit.argtypes = [C.c_void_p, C.c_size_t]
    lib.bp_device_info.argtypes = [C.c_void_p, c_int_p, C.POINTER(C.c_size_t), C.POINTER(C.c_size_t)]
    lib.bp_launch_count.argtypes = [C.c_void_p]
    lib.bp_launch_count.restype = C.c_longlong
    lib.bp_upload_market.argtypes = [C.c_void_p, C.POINTER(MarketDesc)]
    lib.bp_upload_market_async.argtypes = [C.c_void_p, C.POINTER(MarketDesc)]
    lib.bp_prepare_market.argtypes = [C.c_void_p]
    lib.bp_stats_batched.argtypes = [C.c_void_p, C.POINTER(WindowBatchDesc), C.c_void_p, C.c_void_p]
    lib.bp_hf_cov_batched.argtypes = [C.c_void_p, C.POINTER(WindowBatchDesc), C.c_void_p, C.c_void_p]
    lib.bp_conjugate_batched.argtypes = [C.c_void_p, C.POINTER(WindowBatchDesc), C.POINTER(Outputs)]
    lib.bp_jeffreys_batched.argtypes = [C.c_void_p, C.POINTER(WindowBatchDesc), C.POINTER(Outputs)]
    lib.bp_set_stage_timing.argtypes = [C.c_void_p, C.c_int]
    lib.bp_get_stage_times.argtypes = [C.c_void_p, c_double_p, C.POINTER(C.c_longlong)]
    lib.bp_moments_batched.argtypes = [C.c_void_p, C.POINTER(WindowBatchDesc), C.c_int, C.POINTER(Outputs)]
    lib.bp_estimator_batched.argtypes = [C.c_void_p, C.POINTER(WindowBatchDesc), C.c_int, C.POINTER(Outputs)]
    lib.bp_set_resampled.argtypes = [C.c_void_p, C.POINTER(ResampledDesc)]
    lib.bp_get_gram_work.argtypes = [C.c_void_p, c_double_p]
    lib.bp_set_reuse_min_windows.argtypes = [C.c_void_p, C.c_int]
    lib.bp_set_hf_presum_min_days.argtypes = [C.c_void_p, C.c_int]
    lib.bp_set_upload_fractions.argtypes = [C.c_void_p, C.c_int, c_double_p]
    lib.bp_solve_wave_windows.argtypes = [C.c_void_p]
    lib.bp_set_jeffreys_chain.argtypes = [C.c_void_p, C.c_int]
    lib.bp_get_solve_work.argtypes = [C.c_void_p, c_double_p]
    lib.bp_set_condition_estimate.argtypes = [C.c_void_p, C.c_int]
    lib.bp_set_upload_pipeline.argtypes = [C.c_void_p, C.c_int, C.c_longlong]
    lib.bp_set_async_outputs.argtypes = [C.c_void_p, C.c_int]
    lib.bp_backtest_batched.argtypes = [C.c_void_p, C.POINTER(BacktestDesc)]
    lib.bp_excess_returns.argtypes = [C.c_void_p, C.POINTER(WindowBatchDesc), C.c_void_p]
    lib.bp_quadratic_form.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p]
    lib.bp_dense_posterior.argtypes = [C.c_void_p, C.POINTER(DenseProblem), C.POINTER(DenseResult)]
    lib.bp_solve_batched.argtypes = [C.c_void_p, C.POINTER(SolveDesc), C.POINTER(Outputs)]
    for name in EXPORTED:
        getattr(lib, name)          # every declared entry point must be exported
    _lib = lib
    return lib


def last_error() -> str:
    return load().bp_last_error().decode("utf-8", "replace")
