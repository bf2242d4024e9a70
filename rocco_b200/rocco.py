"""Host-side mirror of the hot-path functions of the reference's ``rocco/rocco.py``.

* ``chrom_solution_to_bed`` (rocco.py:139-191), ``_merge_bed_records`` (74-95), ``_write_bed_records``
  (98-110), ``combine_chrom_results`` (194-240): the per-bin Python loop over the mask is replaced by
  run detection on the GPU (``csrc/bed.cu``); text I/O stays on the host.
* ``score_central_tendency_chrom`` (243-304) / ``score_dispersion_chrom`` (307-355): column-wise
  order statistics over the sample axis on the GPU (``csrc/colstats.cu``).
"""
from __future__ import annotations

import ctypes
import logging
import os
from typing import Tuple

import numpy as np

from . import _lib

logger = logging.getLogger(__name__)


def _read_bed_records(bed_file: str) -> tuple[list[tuple[str, int, int]], bool]:
    """(chrom, start, end) of every non-blank line; the flag says whether any line carried more than three columns.
    Lines are stripped, split on tabs, and the coordinates must parse as integers (rocco.py:53-71)."""
    out: list[tuple[str, int, int]] = []
    wide = False
    with open(bed_file, "r", encoding="utf-8") as fh:
        for number, raw in enumerate(fh, start=1):
            cols = raw.strip().split("\t") if raw.strip() else None
            if cols is None:
                continue
            if len(cols) < 3:
                raise ValueError(f"BED row {number} in {bed_file} has fewer than 3 columns.")
            wide |= len(cols) > 3
            out.append((str(cols[0]), int(cols[1]), int(cols[2])))
    return out, wide


def _merge_bed_records(records, min_length_bp: int | None = None):
    """Sort by (chrom STRING, start, end), fuse records that touch or overlap the running interval, then drop the ones
    shorter than ``min_length_bp`` (rocco.py:74-95)."""
    fused: list[list] = []
    for chrom, start, end in sorted(((c, int(s), int(e)) for c, s, e in records), key=lambda r: (r[0], r[1], r[2])):
        if fused and fused[-1][0] == chrom and start <= fused[-1][2]:
            fused[-1][2] = max(fused[-1][2], end)
        else:
            fused.append([chrom, start, end])
    keep = (lambda s, e: True) if min_length_bp is None else (lambda s, e: e - s >= int(min_length_bp))
    return [(str(c), s, e) for c, s, e in fused if keep(s, e)]


def _write_bed_records(records, output_file: str, name_features: bool = False) -> str:
    row = (lambda c, s, e: f"{c}\t{s}\t{e}\t{c}_{s}_{e}\n") if name_features else (lambda c, s, e: f"{c}\t{s}\t{e}\n")
    with open(output_file, "w", encoding="utf-8") as fh:
        fh.write("".join(row(c, s, e) for c, s, e in records))
    return output_file


def solution_runs(solution) -> Tuple[np.ndarray, np.ndarray]:
    """Maximal runs of selected bins among bins 0..n-2 (the last bin is never emitted), on the GPU.

    Returns (first_bin, last_bin + 1) index arrays."""
    sol = np.asarray(solution)
    mask = np.ascontiguousarray(sol if sol.dtype == np.uint8 else (sol > 0.50), dtype=np.uint8)
    if sol.dtype == np.uint8 and mask.max(initial=0) > 1:
        mask = (mask > 0).astype(np.uint8)
    n = mask.shape[0]
    if n == 0:
        return np.zeros(0, np.int64), np.zeros(0, np.int64)
    lib = _lib.load()
    _lib.require_device()
    cap = n // 2 + 1
    starts = np.empty(cap, dtype=np.int64)
    ends = np.empty(cap, dtype=np.int64)
    k = lib.rocco_mask_to_intervals_u8(_lib.np_ptr(mask), n, 0, 1, 0, _lib.np_ptr(starts), _lib.np_ptr(ends), cap)
    if k < 0:
        _lib.check(int(k), "chrom_solution_to_bed")
    return starts[:k], ends[:k]


def chrom_solution_to_bed(chromosome, intervals, solution, ID=None, check_gaps_intervals=True,
                          min_length_bp=None) -> str:
    r"""Convert the decision vector of one chromosome to a BED file in the current directory
    (rocco.py:139-191).  Selected bins (> 0.5) become (intervals[i], intervals[i+1]); the last bin is
    dropped; adjacent records merge; records shorter than ``min_length_bp`` are removed."""
    if len(intervals) != len(solution):
        raise ValueError(
            f"Intervals and solution must have the same length at the pre-merge stage: {len(intervals)} != {len(solution)}")
    intervals_ = np.asarray(intervals)
    if check_gaps_intervals and len(intervals_) > 2:
        # same test as len(set(np.diff(intervals))) > 1 (rocco.py:170-172) without materialising / sorting the differences
        if intervals_.dtype == np.int64 and intervals_.flags.c_contiguous:
            uniform = bool(_lib.load().rocco_b200_uniform_step_i64(_lib.np_ptr(intervals_), len(intervals_)))
        else:
            gaps = np.diff(intervals_)
            uniform = bool(gaps.min() == gaps.max())
        if not uniform:
            raise ValueError(f"Intervals must be contiguous: {set(np.unique(np.diff(intervals_)).tolist())}")
    step_ = intervals_[1] - intervals_[0]  # noqa: F841  (kept: the reference evaluates it, so len < 2 raises)
    output_file = f"rocco_{chromosome}.bed" if ID is None else f"rocco_{ID}_{chromosome}.bed"
    first, last = solution_runs(solution)
    starts = np.asarray(intervals_[first], dtype=np.int64)
    ends = np.asarray(intervals_[last], dtype=np.int64)
    if len(starts) > 1 and not np.all(starts[1:] > ends[:-1]):
        # non-monotone interval tables: full reference merge
        records = _merge_bed_records([(str(chromosome), int(s), int(e)) for s, e in zip(starts.tolist(), ends.tolist())])
        starts = np.array([r[1] for r in records], dtype=np.int64)
        ends = np.array([r[2] for r in records], dtype=np.int64)
    if min_length_bp is not None:
        keep = (ends - starts) >= int(min_length_bp)
        starts, ends = starts[keep], ends[keep]
    return _lib.write_bed_arrays(output_file, [str(chromosome)], None, starts, ends)


def combine_chrom_results(chrom_bed_files: list, output_file: str, name_features: bool = False) -> str:
    r"""Concatenate per-chromosome BED files, sort by (chrom string, start, end), merge, write (rocco.py:194-240).

    Canonical BED text (what this package and the reference write) is read, sorted, merged and written in one native
    pass; anything the native parser declines (ragged rows, stray whitespace, non-integer coordinates, ...) goes through
    the line-by-line reader above, whose tolerance and error messages are the reference's."""
    if os.path.exists(output_file):
        logger.info(f"Removing existing output file: {output_file}")
        try:
            os.remove(output_file)
        except OSError:
            logger.info(f"Could not remove existing output file: {output_file}.")
    for f in chrom_bed_files:
        if not os.path.exists(f):
            raise FileNotFoundError(f"File does not exist: {f}")
    extra_msg = "More than 3 columns detected in the input BED files. Extra columns will be ignored."
    native = _lib.combine_bed_files(list(chrom_bed_files), output_file, name_features) if len(chrom_bed_files) else None
    if native is not None:
        if native[1]:
            logger.info(extra_msg)
        return output_file
    records, told = [], False
    for f in chrom_bed_files:
        try:
            recs, wide = _read_bed_records(f)
        except Exception as e:
            logger.info(f"Could not read BED file: {f}\n{e}\n")
            raise
        if wide and not told:
            logger.info(extra_msg)
            told = True
        records.extend(recs)
    return _write_bed_records(_merge_bed_records(records), output_file, name_features=name_features)


# ------------------------------------------------------------------------------------------------
# column-wise statistics over the sample axis (rocco.py:243-355)
# ------------------------------------------------------------------------------------------------
_STAT = {"median": 0, "quantile": 1, "tmean": 2, "mean": 3, "mad": 4, "iqr": 5, "std": 6, "tstd": 7}


def _column_stat(chrom_matrix: np.ndarray, stat: str, arg0: float = 0.0, arg1: float = 0.0, power: float = 1.0) -> np.ndarray:
    x = np.ascontiguousarray(chrom_matrix, dtype=np.float64)
    m, n = x.shape
    out = np.zeros(n, dtype=np.float64)
    if n == 0:
        return out
    lib = _lib.load()
    _lib.require_device()
    st = lib.rocco_column_stat_f64(_lib.np_ptr(x), m, n, _STAT[stat], float(arg0), float(arg1), float(power), _lib.np_ptr(out))
    _lib.check(st, "column statistic")
    return out


def _normalize_method(method) -> str:
    return str(method).strip().lower().replace("-", "").replace("_", "")


def _central_tendency_stat(method, quantile=0.50, tprop=0.05) -> tuple[str, float, float]:
    """(statistic, arg0, arg1) of a ``score_central_tendency_chrom`` method with its arguments."""
    method_ = _normalize_method(method)
    if method_ == "quantile":
        if not 0.0 <= quantile <= 1.0:
            logger.warning("`quantile` must be in [0, 1]. Using the median instead.")
            quantile = 0.50
        if quantile == 0.50:
            return "median", 0.0, 0.0
        return "quantile", quantile, 0.0
    if method_ == "tmean":
        return "tmean", tprop, 0.0
    if method_ == "mean":
        return "mean", 0.0, 0.0
    raise ValueError(f"Central tendency method not recognized: {method}")


def _dispersion_stat(method, rng=(25, 75), tprop=0.05) -> tuple[str, float, float]:
    """(statistic, arg0, arg1) of a ``score_dispersion_chrom`` method with its arguments."""
    method_ = _normalize_method(method)
    if method_ == "mad":
        return "mad", 0.0, 0.0
    if method_ == "iqr":
        return "iqr", rng[0], rng[1]
    if method_ == "std":
        return "std", 0.0, 0.0
    if method_ == "tstd":
        return "tstd", tprop, 0.0
    raise ValueError(f"Dispersion method not recognized or could not execute: {method}")


def score_central_tendency_chrom(chrom_matrix, method="quantile", quantile=0.50, tprop=0.05, power=1.0) -> np.ndarray:
    r"""Return a column-wise location summary across samples (rocco.py:243-304)."""
    chrom_matrix = np.asarray(chrom_matrix, dtype=float)
    if chrom_matrix.ndim != 2:
        raise ValueError("`chrom_matrix` must be a 2D array.")
    if chrom_matrix.shape[0] == 1:
        return _column_stat(chrom_matrix, "mean", power=power)
    stat, arg0, arg1 = _central_tendency_stat(method, quantile, tprop)
    return _column_stat(chrom_matrix, stat, arg0=arg0, arg1=arg1, power=power)


def score_dispersion_chrom(chrom_matrix: np.ndarray, method: str = "mad", rng: Tuple[int, int] = (25, 75),
                           tprop: float = 0.05, power: float = 1.0) -> np.ndarray:
    r"""Return a column-wise dispersion summary across samples (rocco.py:307-355).

    ``tstd`` computes the evident per-column intent -- sample standard deviation (ddof 1) of the values
    inside the inclusive nearest-rank limits; the reference itself raises for that method under current
    SciPy (SURVEY.md section 8a row a7)."""
    chrom_matrix = np.asarray(chrom_matrix, dtype=float)
    if chrom_matrix.ndim != 2:
        raise ValueError("`chrom_matrix` must be a 2D array.")
    if chrom_matrix.shape[0] == 1:
        return _column_stat(chrom_matrix, "mad", power=power)
    stat, arg0, arg1 = _dispersion_stat(method, rng, tprop)
    return _column_stat(chrom_matrix, stat, arg0=arg0, arg1=arg1, power=power)


# ------------------------------------------------------------------------------------------------
# automatic gamma (rocco.py:751-789) -- SURVEY.md 8(f) rank 2
# ------------------------------------------------------------------------------------------------
def _resolve_chrom_gamma(chrom: str, args: dict, chrom_scores: np.ndarray, budget_rate_meta: dict) -> tuple[float, dict | None]:
    r"""gamma = clip(0.5 * ceil(tau_int) * median(scores > 0), 0.5, 10) unless ``args["gamma"]`` fixes it.

    The median of the positive scores is taken on the GPU; when ``budget_rate_meta`` comes from this package's budget
    estimator it already carries that number (computed while the scores were on the device) and nothing is re-read."""
    if args["gamma"] is not None:
        chrom_gamma = float(args["gamma"])
        if not np.isfinite(chrom_gamma) or chrom_gamma < 0.0:
            raise ValueError("`--gamma` must be finite and non-negative")
        logger.info("%s fixed gamma value=%.6f", chrom, chrom_gamma)
        return float(chrom_gamma), None
    if "positive_score_median" in budget_rate_meta and "positive_score_count" in budget_rate_meta:
        positive_scale = float(budget_rate_meta["positive_score_median"])
        positive_count = int(budget_rate_meta["positive_score_count"])
    else:
        scores_ = np.ascontiguousarray(chrom_scores, dtype=np.float64)
        med, cnt = ctypes.c_double(1.0), ctypes.c_longlong(0)
        if scores_.size:
            _lib.require_device()
            _lib.check(_lib.load().rocco_positive_score_median_f64(_lib.np_ptr(scores_), scores_.size, ctypes.byref(med),
                                                                   ctypes.byref(cnt)), "positive score median")
        positive_scale, positive_count = float(med.value), int(cnt.value)
    autocorrelation_time = max(1.0, float(budget_rate_meta.get("autocorrelation_time", 1.0)))
    characteristic_run = int(np.ceil(autocorrelation_time))
    gamma_raw = 0.5 * float(characteristic_run) * float(positive_scale)
    chrom_gamma = float(np.clip(gamma_raw, 0.5, 10.0))
    gamma_meta = {
        "method": "auto_score_autocorr", "autocorrelation_time": float(autocorrelation_time),
        "characteristic_run_length": int(characteristic_run), "positive_score_median": float(positive_scale),
        "positive_score_count": int(positive_count), "gamma_raw": float(gamma_raw), "gamma_clipped": float(chrom_gamma),
        "gamma_clip_min": 0.5, "gamma_clip_max": 10.0,
    }
    logger.info("%s auto gamma estimate: %s", chrom, gamma_meta)
    return float(chrom_gamma), gamma_meta


# ------------------------------------------------------------------------------------------------
# chromosome budgets for the solves (rocco.py:1113-1143) -- SURVEY.md 8(f) rank 2
# ------------------------------------------------------------------------------------------------
def _resolve_budgets(chrom_cache: dict, args: dict) -> tuple[dict, dict]:
    r"""EB-shrunk per-chromosome budgets from the cached budget estimates, rescaled so that the prior centre lands on
    ``args["budget"]`` when that is given, times ``args["scale_chrom_budgets"]``, clipped to [0.005, 0.1]."""
    from .inference import estimate_empirical_bayes_budgets
    candidates = {c: chrom_cache[c]["budget_count_hat"] for c in chrom_cache}
    totals = {c: chrom_cache[c]["total_count"] for c in chrom_cache}
    shrunk, budget_meta = estimate_empirical_bayes_budgets(candidates, totals, posterior_quantile=args["budget_posterior_quantile"])
    centre = budget_meta["genome_wide_budget"]
    to_target = float(args["budget"]) / centre if (args["budget"] is not None and centre > 0) else 1.0
    user_scale = float(args["scale_chrom_budgets"])
    # (budget * rescale) * scale: the reference's association order, kept so the doubles agree
    chrom_budgets = {c: min(max(b * to_target * user_scale, 0.005), 0.1) for c, b in shrunk.items()}
    logger.info("Empirical-Bayes budget prior: %s", budget_meta)
    return chrom_budgets, budget_meta


# ------------------------------------------------------------------------------------------------
# narrowPeak summit offsets (rocco.py:809-872) -- SURVEY.md 8(f) rank 4
# ------------------------------------------------------------------------------------------------
def _cpy_narrowpeak_summit_track(chrom: str, intervals: np.ndarray, effect_mean: np.ndarray) -> str | None:
    r"""Park (bin starts, bin centres, float32 WLS mean) of one chromosome in a temporary ``.npz`` (rocco.py:809-837);
    host-side I/O only."""
    import tempfile
    intervals_ = np.asarray(intervals, dtype=np.int64)
    effect_mean_ = np.asarray(effect_mean, dtype=np.float32)
    usable = int(min(max(intervals_.shape[0] - 1, 0), effect_mean_.shape[0]))
    if usable <= 0:
        return None
    fd, summit_track_file = tempfile.mkstemp(prefix=f"rocco_summit_track_{chrom}_", suffix=".npz")
    os.close(fd)
    np.savez(summit_track_file, starts=intervals_[:usable], centers=(intervals_[:usable] + intervals_[1:usable + 1]) // 2,
             mean=effect_mean_[:usable])
    return summit_track_file


def narrowpeak_summit_offsets(track_starts, track_centers, track_mean, peak_starts, peak_ends) -> np.ndarray:
    """Summit offset of every peak of one chromosome (segmented arg-max of the mean on the GPU); -1 where the reference
    writes -1."""
    ps = np.ascontiguousarray(peak_starts, dtype=np.int64)
    pe = np.ascontiguousarray(peak_ends, dtype=np.int64)
    out = np.full(ps.shape[0], -1, dtype=np.int64)
    if ps.shape[0] == 0:
        return out
    ts = np.ascontiguousarray(track_starts, dtype=np.int64)
    tc = np.ascontiguousarray(track_centers, dtype=np.int64)
    tm = np.ascontiguousarray(track_mean, dtype=np.float32)
    _lib.require_device()
    _lib.check(_lib.load().rocco_narrowpeak_summit_offsets_f32(_lib.np_ptr(ts), _lib.np_ptr(tc), _lib.np_ptr(tm), ts.shape[0],
                                                               _lib.np_ptr(ps), _lib.np_ptr(pe), ps.shape[0], _lib.np_ptr(out)),
               "narrowPeak summit offsets")
    return out


def _write_narrowpeak_summit_offsets(peak_file: str, chrom_cache: dict, output_file: str) -> str:
    r"""``<chrom>_<start>_<end>\t<summit offset>`` for every record of ``peak_file`` (rocco.py:840-872); the arg-max over
    each peak runs on the GPU, one launch per chromosome."""
    records, _ = _read_bed_records(peak_file)
    offsets = np.full(len(records), -1, dtype=np.int64)
    by_chrom: dict[str, list[int]] = {}
    for k, (chrom, _s, _e) in enumerate(records):
        by_chrom.setdefault(chrom, []).append(k)
    for chrom, idx in by_chrom.items():
        summit_track_file = chrom_cache.get(chrom, {}).get("summit_track_file")
        if summit_track_file is None:
            continue
        with np.load(summit_track_file) as summit_track:
            starts = np.asarray(summit_track["starts"], dtype=np.int64)
            centers = np.asarray(summit_track["centers"], dtype=np.int64)
            mean_track = np.asarray(summit_track["mean"], dtype=np.float32)
        offsets[idx] = narrowpeak_summit_offsets(starts, centers, mean_track, [records[k][1] for k in idx],
                                                 [records[k][2] for k in idx])
    with open(output_file, "w", encoding="utf-8") as handle:
        handle.write("".join(f"{c}_{s}_{e}\t{int(o)}\n" for (c, s, e), o in zip(records, offsets)))
    return output_file
