"""ctypes binding of ``librocco_b200.so`` (the C-ABI declared in ``include/rocco_b200.h``).

There is no CPU fallback anywhere in this package: if the shared library is missing or no CUDA
device is visible, every compute entry raises ``RuntimeError`` -- mirroring the reference's
"Make sure native C extensions are built and available" (dp.py:73-74, inference.py:244-245).
"""
from __future__ import annotations

import ctypes
import os
from ctypes import POINTER, Structure, c_char_p, c_double, c_int, c_longlong, c_size_t, c_ubyte, c_ulonglong, c_void_p

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "librocco_b200.so")

ST_NOMEM, ST_INVALID, ST_CUDA, ST_NONFINITE = -1, -2, -3, -4


class ChainResult(Structure):
    _fields_ = [
        ("selection_penalty", c_double), ("penalized_objective", c_double), ("objective", c_double),
        ("selected_count", c_longlong), ("switch_count", c_longlong), ("exact_tie_bins", c_longlong),
        ("near_tie_bins", c_longlong), ("dp_passes", c_int), ("search_rounds", c_int),
        ("status", c_int), ("reserved", c_int),
    ]


class ChainTask(Structure):
    _fields_ = [
        ("offset", c_size_t), ("n", c_size_t), ("gamma", c_double), ("cost_sum", c_double),
        ("selection_penalty", c_double), ("target_count", c_longlong), ("mode", c_int), ("max_iter", c_int),
    ]


class GenomeSearch(Structure):
    _fields_ = [
        ("total_bins", c_longlong), ("target_count", c_longlong), ("cost_sum", c_double), ("cost_max", c_double),
        ("score_min", c_double), ("score_max", c_double), ("max_iter", c_int), ("reserved", c_int),
    ]


class GenomeResult(Structure):
    _fields_ = [
        ("selection_penalty", c_double), ("selected_count", c_longlong), ("dp_passes", c_int), ("search_rounds", c_int),
        ("status", c_int), ("reserved", c_int),
    ]


class ScoreParams(Structure):
    _fields_ = [
        ("lower_bound_z", c_double), ("prior_df", c_double), ("min_effect", c_double),
        ("use_min_effect", c_int), ("spatial_window", c_int), ("precision_floor_ratio", c_double),
        ("baseline_window", c_int), ("pilot_mode", c_int),
    ]


class ScoreOutputs(Structure):
    _fields_ = [
        ("scores", c_void_p), ("mean", c_void_p), ("raw_variance", c_void_p), ("prior_variance", c_void_p),
        ("moderated_variance", c_void_p), ("standard_error", c_void_p), ("centered_matrix", c_void_p),
        ("total_df", c_double), ("resolved_spatial_window", c_int), ("baseline_window", c_int),
        ("baseline_lambda", c_double),
    ]


class BudgetParams(Structure):
    _fields_ = [
        ("score", ScoreParams), ("dependence_lag_hint", c_int), ("num_null_draws", c_int), ("min_null_draws", c_int),
        ("sample_offset", c_int), ("stability_abs_tol", c_double), ("stability_rel_tol", c_double),
        ("random_seed", c_ulonglong), ("d_innovations", c_void_p), ("random_streams", c_int),
    ]


# rocco_b200_allreduce_fn: sum d_buf[0:count) over ranks in place, stream-ordered; 0 = success
ALLREDUCE_FN = ctypes.CFUNCTYPE(c_int, c_void_p, c_size_t, c_void_p, c_void_p)


_BUDGET_DOUBLES = (
    "nonnull_fraction", "effective_count", "effective_total_count", "autocorrelation_time", "null_center", "null_scale",
    "null_threshold", "null_positive_mass", "null_positive_units", "null_positive_fraction", "null_positive_units_sd",
    "null_positive_units_stderr", "null_tail_occupancy", "null_tail_occupancy_sd", "null_tail_occupancy_stderr",
    "negative_fraction", "observed_positive_fraction", "observed_negative_fraction", "observed_excess_mass",
    "observed_excess_units", "observed_tail_occupancy", "null_reference_mean_positive_consensus",
    "null_reference_max_positive_consensus", "positive_score_median")
_BUDGET_LONGS = ("negative_support_size", "positive_score_count", "num_loci")
_BUDGET_INTS = ("num_null_draws", "max_null_draws", "adaptive_stop", "wild_bandwidth", "ess_max_lag", "ess_lags_used")


class BudgetResult(Structure):
    _fields_ = ([(k, c_double) for k in _BUDGET_DOUBLES] + [(k, c_longlong) for k in _BUDGET_LONGS]
                + [(k, c_int) for k in _BUDGET_INTS])


class CountOptions(Structure):
    _fields_ = [
        ("flag_include", ctypes.c_int32), ("flag_exclude", ctypes.c_int32), ("min_mapping_quality", ctypes.c_int32),
        ("paired_end_mode", ctypes.c_int32), ("one_read_per_bin", ctypes.c_int32), ("reserved", ctypes.c_int32),
        ("read_length", ctypes.c_int64), ("min_template_length", ctypes.c_int64), ("max_insert_size", ctypes.c_int64),
        ("shift_forward_strand53", ctypes.c_int64), ("shift_reverse_strand53", ctypes.c_int64), ("extend_bp", ctypes.c_int64),
    ]


class Track(Structure):
    _fields_ = [
        ("d_counts", c_void_p), ("count_len", c_size_t), ("count_start", ctypes.c_int64), ("norm_scale", c_double),
        ("const_scale", c_double), ("scale_by_step", ctypes.c_int32), ("reserved", ctypes.c_int32),
    ]


_lib = None


def _declare(lib):
    dp, u8p, llp, ip = POINTER(c_double), POINTER(c_ubyte), POINTER(c_longlong), POINTER(c_int)
    sig = {
        "rocco_b200_version": (c_char_p, []),
        "rocco_b200_last_error": (c_char_p, []),
        "rocco_b200_device_count": (c_int, []),
        "rocco_b200_set_device": (c_int, [c_int]),
        "rocco_b200_kernel_launches": (c_ulonglong, []),
        "rocco_b200_profile_enable": (c_int, [c_int]),
        "rocco_b200_profile_report": (c_int, [c_char_p, c_size_t]),
        "rocco_b200_profile_timeline": (c_int, [c_char_p, c_size_t]),
        "rocco_b200_uniform_step_i64": (c_int, [c_void_p, c_size_t]),
        "rocco_b200_write_bed3": (c_int, [c_char_p, POINTER(c_char_p), c_int, c_void_p, c_void_p, c_void_p, c_size_t, c_int]),
        "rocco_b200_write_bed3_at": (c_int, [c_char_p, c_longlong, POINTER(c_char_p), c_int, c_void_p, c_void_p, c_void_p, c_size_t, c_int,
                                     POINTER(c_longlong)]),
        "rocco_b200_combine_bed3": (ctypes.c_longlong, [POINTER(c_char_p), c_int, c_char_p, c_int, POINTER(c_int)]),
        "rocco_b200_default_budget_params": (None, [POINTER(BudgetParams)]),
        "rocco_b200_budget_bandwidth": (c_int, [c_size_t, c_int]),
        "rocco_b200_budget_ess_max_lag": (c_int, [c_size_t, c_int]),
        "rocco_b200_budget_nonnull_fraction_dev": (c_int, [c_void_p, c_size_t, c_size_t, c_void_p, POINTER(BudgetParams),
                                                           POINTER(BudgetResult), c_void_p]),
        "rocco_b200_budget_nonnull_fraction_sharded_dev": (
            c_int, [c_void_p, c_size_t, c_size_t, c_size_t, c_void_p, POINTER(BudgetParams), c_void_p, c_void_p,
                    POINTER(BudgetResult), c_void_p]),
        "rocco_budget_nonnull_fraction_f64": (c_int, [c_void_p, c_size_t, c_size_t, c_void_p, POINTER(BudgetParams), c_void_p,
                                                      POINTER(BudgetResult)]),
        "rocco_b200_wild_multiply_dev": (c_int, [c_void_p, c_size_t, c_size_t, c_int, c_ulonglong, ctypes.c_uint, c_void_p, c_void_p,
                                                 c_void_p]),
        "rocco_b200_numpy_normals_dev": (c_int, [c_ulonglong, c_ulonglong, c_ulonglong, c_ulonglong, c_void_p,
                                                 POINTER(c_ulonglong), c_void_p]),
        "rocco_b200_numpy_seed_state": (c_int, [c_ulonglong, c_ulonglong, POINTER(c_ulonglong)]),
        "rocco_b200_numpy_streams_set_chunk_words": (c_int, [c_int]),
        "rocco_effective_sample_size_f64": (c_int, [c_void_p, c_size_t, c_int, dp, dp, ip]),
        "rocco_positive_score_median_f64": (c_int, [c_void_p, c_size_t, dp, llp]),
        "rocco_b200_pull_pinned": (c_int, [c_void_p, c_void_p, c_size_t, c_void_p]),
        "rocco_narrowpeak_summit_offsets_f32": (c_int, [c_void_p, c_void_p, c_void_p, c_size_t, c_void_p, c_void_p, c_size_t, c_void_p]),
        "rocco_b200_summit_offsets_dev": (c_int, [c_void_p, c_void_p, c_void_p, c_size_t, c_void_p, c_void_p, c_size_t, c_void_p, c_void_p]),
        "rocco_b200_numpy_sum_f64": (c_double, [c_void_p, c_size_t]),
        "rocco_b200_numpy_sum_const_f64": (c_double, [c_double, c_size_t]),
        "rocco_solve_penalized_chain_f64": (c_int, [c_void_p, c_void_p, c_size_t, c_double, c_void_p, dp, llp]),
        "rocco_calibrate_selection_penalty_f64": (
            c_int, [c_void_p, c_void_p, c_size_t, c_longlong, c_int, dp, c_void_p, dp, llp]),
        "rocco_b200_chain_solve_batch_dev": (
            c_int, [c_void_p, c_void_p, POINTER(ChainTask), c_int, c_void_p, POINTER(ChainResult), c_int, c_void_p]),
        "rocco_b200_chain_solve_genome_dev": (
            c_int, [c_void_p, c_void_p, POINTER(ChainTask), c_int, POINTER(GenomeSearch), c_void_p, c_void_p, c_void_p,
                    POINTER(ChainResult), POINTER(GenomeResult), c_int, c_void_p]),
        "rocco_b200_chain_set_seq_max": (c_int, [c_int]),
        "rocco_b200_chain_set_exact_search": (c_int, [c_int]),
        "rocco_b200_chain_set_tile_freezing": (c_int, [c_int]),
        "rocco_b200_chain_sweep_dev": (
            c_int, [c_void_p, c_size_t, c_double, c_void_p, c_int, c_void_p, c_void_p, c_void_p, c_void_p]),
        "rocco_mask_to_intervals_u8": (
            c_longlong, [c_void_p, c_size_t, c_longlong, c_longlong, c_longlong, c_void_p, c_void_p, c_size_t]),
        "rocco_b200_mask_to_intervals_dev": (
            c_longlong, [c_void_p, c_size_t, c_longlong, c_longlong, c_longlong, c_void_p, c_void_p, c_size_t, c_void_p]),
        "rocco_b200_mask_to_runs_batch_dev": (
            c_longlong, [c_void_p, c_void_p, c_void_p, c_int, c_void_p, c_void_p, c_void_p, c_size_t, c_void_p]),
        "rocco_crossfit_whittaker_baseline_f64": (c_int, [c_void_p, c_size_t, c_double, c_void_p]),
        "rocco_crossfit_whittaker_baseline_matrix_f64": (c_int, [c_void_p, c_size_t, c_size_t, c_double, c_void_p]),
        "rocco_score_centered_wls_f64": (
            c_int, [c_void_p, c_size_t, c_size_t, c_double, c_double, c_double, c_int, c_int, c_double,
                    c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, dp, ip]),
        "rocco_b200_default_score_params": (None, [POINTER(ScoreParams)]),
        "rocco_b200_trim_pools": (c_int, [c_size_t]),
        "rocco_b200_trend_set_mode": (c_int, [c_int]),
        "rocco_b200_trend_fallback_rows": (c_longlong, []),
        "rocco_b200_trend_fallback_reasons": (None, [c_void_p]),
        "rocco_b200_whittaker_exact_rows": (c_longlong, []),
        "rocco_score_loci_wls_f64": (c_int, [c_void_p, c_size_t, c_size_t, POINTER(ScoreParams), POINTER(ScoreOutputs)]),
        "rocco_score_loci_wls_f32": (c_int, [c_void_p, c_size_t, c_size_t, POINTER(ScoreParams), POINTER(ScoreOutputs)]),
        "rocco_b200_score_loci_wls_dev": (
            c_int, [c_void_p, c_int, c_size_t, c_size_t, POINTER(ScoreParams), POINTER(ScoreOutputs), c_void_p]),
        "rocco_b200_score_partial_dev": (c_int, [c_void_p, c_int, c_size_t, c_size_t, POINTER(ScoreParams), c_void_p, c_void_p]),
        "rocco_b200_score_partial_ex_dev": (
            c_int, [c_void_p, c_int, c_size_t, c_size_t, POINTER(ScoreParams), c_void_p, c_void_p, c_void_p]),
        "rocco_b200_score_finalize_dev": (c_int, [c_void_p, c_size_t, c_size_t, POINTER(ScoreParams), POINTER(ScoreOutputs), c_void_p]),
        "rocco_b200_crossfit_baseline_dev": (c_int, [c_void_p, c_size_t, c_size_t, c_double, c_void_p, c_void_p]),
        "rocco_b200_score_centered_wls_dev": (
            c_int, [c_void_p, c_size_t, c_size_t, POINTER(ScoreParams), POINTER(ScoreOutputs), c_void_p]),
        "rocco_b200_count_alignment_region_dev": (
            c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_size_t, POINTER(CountOptions), ctypes.c_int64,
                    ctypes.c_int64, ctypes.c_int64, c_void_p, c_size_t, c_void_p]),
        "rocco_b200_track_positive_range_dev": (c_int, [POINTER(Track), c_int, ctypes.c_int64, c_void_p, c_void_p, c_void_p]),
        "rocco_b200_assemble_matrix_dev": (
            c_int, [POINTER(Track), c_void_p, c_void_p, c_int, ctypes.c_int64, c_int, c_void_p, c_void_p, c_int, c_size_t, c_int,
                    c_void_p, c_void_p, c_void_p]),
        "rocco_column_stat_f64": (c_int, [c_void_p, c_size_t, c_size_t, c_int, c_double, c_double, c_double, c_void_p]),
        "rocco_b200_column_stat_dev": (
            c_int, [c_void_p, c_int, c_size_t, c_size_t, c_int, c_double, c_double, c_double, c_void_p, c_void_p]),
        "rocco_b200_colstat_set_mode": (c_int, [c_int]),
    }
    for name, (res, args) in sig.items():
        fn = getattr(lib, name)          # AttributeError here = header/library mismatch: fail loudly
        fn.restype = res
        fn.argtypes = args
    return sig


def load():
    """Load (once) and return the shared library; raises RuntimeError when it has not been built."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(
                f"{LIB_PATH} not found. Make sure native CUDA extensions are built and available "
                "(python -c 'import __graft_entry__ as g; g.build()' or make -C rocco_b200/csrc).")
        lib = ctypes.CDLL(LIB_PATH)
        lib._signatures = _declare(lib)
        _lib = lib
    return _lib


def last_error() -> str:
    return load().rocco_b200_last_error().decode("utf-8", "replace")


def check(status: int, what: str = "rocco_b200") -> None:
    """Map C-ABI status codes onto the reference's exceptions (_wls.c:133-150, _baseline.c:96-101)."""
    if status == 0:
        return
    if status == ST_NOMEM:
        raise MemoryError(f"{what}: device/host allocation failed ({last_error()})")
    if status == ST_INVALID:
        raise ValueError(f"{what}: invalid inputs")
    if status == ST_NONFINITE:
        raise ValueError(f"{what}: non-finite values")
    raise RuntimeError(f"{what}: CUDA error: {last_error()}")


_CUDA_PID = None


def require_device() -> None:
    """Every compute entry passes through here first.  The reference runs its native kernels from FORKED worker pools
    (rocco.py:1176-1180, inference.py:871-893); a CUDA context does not survive a fork, and the driver's own message for that
    is an opaque "initialization error", so the situation is named here instead."""
    global _CUDA_PID
    pid = os.getpid()
    if _CUDA_PID is not None and _CUDA_PID != pid:
        raise RuntimeError(
            f"rocco_b200: the CUDA context was created in process {_CUDA_PID}; this forked child ({pid}) cannot use it. "
            "Drive chromosomes from threads (each call leases its own stream), start workers with the 'spawn' method, or pass "
            "all chromosomes to one call (rocco_b200.pipeline.solve_chromosomes / run_shard).")
    if load().rocco_b200_device_count() <= 0:
        raise RuntimeError("rocco_b200: no CUDA device visible and there is no CPU fallback")
    _CUDA_PID = pid


def np_ptr(a: np.ndarray) -> c_void_p:
    return c_void_p(a.ctypes.data)


def trim_pools(bytes_to_keep: int = 0) -> int:
    """Hand the scratch cached in the library's CUDA memory pools (beyond ``bytes_to_keep`` per pool) back to the driver."""
    return int(load().rocco_b200_trim_pools(int(bytes_to_keep)))


def kernel_launches() -> int:
    return int(load().rocco_b200_kernel_launches())


def numpy_sum_const(value: float, n: int) -> float:
    """numpy.sum(numpy.full(n, value)) without materialising the vector (dp.py:110-111 bracket)."""
    return float(load().rocco_b200_numpy_sum_const_f64(float(value), int(n)))


def profile_enable(on: bool) -> bool:
    return bool(load().rocco_b200_profile_enable(1 if on else 0))


def profile_report() -> dict:
    """{scope: (total_ms, launch_sets, algorithmic_bytes)} since the last report; synchronises the device."""
    buf = ctypes.create_string_buffer(1 << 16)
    load().rocco_b200_profile_report(buf, len(buf))
    out = {}
    for line in buf.value.decode().splitlines():
        name, ms, cnt, nbytes = line.split()
        out[name] = (float(ms), int(cnt), float(nbytes))
    return out


def profile_timeline() -> list:
    """[(scope, start_ms, duration_ms)] of the scopes recorded since the last report, in record order."""
    buf = ctypes.create_string_buffer(1 << 22)
    load().rocco_b200_profile_timeline(buf, len(buf))
    return [(a, float(b), float(c)) for a, b, c in (line.split() for line in buf.value.decode().splitlines())]


def write_bed_arrays(path: str, names, name_idx, starts: np.ndarray, ends: np.ndarray, name_features: bool = False) -> str:
    """BED3/BED4 text of (names[name_idx[i]], starts[i], ends[i]) written by the native formatter."""
    lib = load()
    starts = np.ascontiguousarray(starts, dtype=np.int64)
    ends = np.ascontiguousarray(ends, dtype=np.int64)
    arr = (c_char_p * len(names))(*[str(x).encode("utf-8") for x in names])
    idx = None if name_idx is None else np.ascontiguousarray(name_idx, dtype=np.int32)
    st = lib.rocco_b200_write_bed3(str(path).encode("utf-8"), arr, len(names), None if idx is None else np_ptr(idx),
                                   np_ptr(starts), np_ptr(ends), len(starts), 1 if name_features else 0)
    if st != 0:
        raise OSError(f"could not write BED file {path}: {last_error()}")
    return path


def write_bed_arrays_at(path: str, offset: int, names, name_idx, starts: np.ndarray, ends: np.ndarray, name_features: bool = False) -> int:
    """The text of write_bed_arrays placed at byte `offset` of `path` (no truncation); returns the number of bytes written."""
    lib = load()
    starts = np.ascontiguousarray(starts, dtype=np.int64)
    ends = np.ascontiguousarray(ends, dtype=np.int64)
    arr = (c_char_p * len(names))(*[str(x).encode("utf-8") for x in names])
    idx = None if name_idx is None else np.ascontiguousarray(name_idx, dtype=np.int32)
    written = c_longlong(0)
    st = lib.rocco_b200_write_bed3_at(str(path).encode("utf-8"), int(offset), arr, len(names), None if idx is None else np_ptr(idx),
                                      np_ptr(starts), np_ptr(ends), len(starts), 1 if name_features else 0, ctypes.byref(written))
    if st != 0:
        raise OSError(f"could not write BED file {path}: {last_error()}")
    return int(written.value)


def combine_bed_files(paths, output_file: str, name_features: bool = False):
    """Native combine of canonical BED files; returns (records_written, saw_extra_columns) or None when a file needs the
    line-by-line reader."""
    lib = load()
    arr = (c_char_p * len(paths))(*[os.fsencode(str(x)) for x in paths])
    extra = c_int(0)
    n = lib.rocco_b200_combine_bed3(arr, len(paths), os.fsencode(str(output_file)), 1 if name_features else 0, ctypes.byref(extra))
    if n == -1:
        return None
    if n < 0:
        raise OSError(f"could not write BED file {output_file}: {last_error()}")
    return int(n), bool(extra.value)
