"""Host-side mirror of the scoring half of the reference's ``rocco/inference.py`` (lines 32-379).

Same function names, arguments, return types and exceptions.  ``score_loci_wls`` runs the whole
chain (log2p1 -> pilot offset -> cross-fit Whittaker baseline -> centered WLS) in one C-ABI call so the
reference's four m x n float64 temporaries (inference.py:325-341) never exist on the host; the stage
functions are kept for callers (and tests) that use them on their own.
"""
from __future__ import annotations

import ctypes
import logging
from typing import Any, Dict, Tuple

import numpy as np

from . import _baseline as _baseline_native
from . import _lib
from . import _wls as _wls_native
from .pipeline import score_params

logger = logging.getLogger(__name__)


def _finite_or_raise(what: str, *arrays) -> None:
    for a in arrays:
        if not np.isfinite(a).all():
            raise ValueError(what)


def _log_scale_wls_matrix(chrom_matrix: np.ndarray, pseudocount: float = 1.0) -> np.ndarray:
    """log2(max(x, 0) + pseudocount) in float64; non-finite input is an error (inference.py:40-47)."""
    x = np.asarray(chrom_matrix, dtype=np.float64)
    _finite_or_raise("`chrom_matrix` contains non-finite values", x)
    return np.log2(np.maximum(x, 0.0) + float(pseudocount))


def _resolve_local_baseline_window(n_loci: int, target_window: int = 101) -> int:
    """Odd window <= n for the Whittaker baseline, 0 for rows shorter than 25 bins (inference.py:50-62)."""
    n = int(n_loci)
    if n < 25:
        return 0
    w = min(max(3, int(target_window)), n)
    if w % 2 == 0:                      # force odd: shrink only when the window already spans the row
        w += -1 if w == n else 1
    return max(0, w)


def _consenrich_whittaker_lambda(block_size: int) -> float:
    """lambda = 7 (w / 2 pi)^4 for an odd block w >= 3 (inference.py:65-76; 0.15915494 is the reference's 1 / 2 pi)."""
    w = max(3, int(block_size))
    w += 1 - (w % 2)
    return float(7.0 * (float(w) * 0.15915494) ** 4)


def _consenrich_crossfit_whittaker_baseline(y_vals: np.ndarray, block_size: int = 101) -> np.ndarray:
    y = np.asarray(y_vals, dtype=np.float64)
    if y.ndim != 1:
        raise ValueError("`y_vals` must be one-dimensional")
    w = _resolve_local_baseline_window(y.size, target_window=block_size)
    if w == 0:
        return np.zeros_like(y)
    return np.asarray(_baseline_native.crossfit_whittaker_baseline(y, penalty_lambda=_consenrich_whittaker_lambda(w)), dtype=np.float64)


def _estimate_local_background_matrix(centered_matrix: np.ndarray, target_window: int = 101) -> tuple[np.ndarray, int, float]:
    """Row-wise cross-fit Whittaker baseline: (baselines, resolved window, lambda) (inference.py:185-228)."""
    rows = np.asarray(centered_matrix, dtype=np.float64)
    if rows.ndim != 2:
        raise ValueError("`centered_matrix` must be two-dimensional")
    w = _resolve_local_baseline_window(rows.shape[1], target_window=target_window)
    if w == 0:
        return np.zeros_like(rows), 0, 0.0
    lam = _consenrich_whittaker_lambda(w)
    base = np.asarray(_baseline_native.crossfit_whittaker_baseline(rows, penalty_lambda=lam), dtype=np.float64)
    _finite_or_raise("Local baseline fit produced non-finite values", base)
    return base, w, lam


_WLS_FIELDS = ("mean", "raw_variance", "prior_variance", "moderated_variance", "standard_error")


def _score_centered_wls_matrix(centered_matrix: np.ndarray, lower_bound_z: float = 1.0, prior_df: float = 5.0,
                               min_effect: float | None = None, spatial_window: int | None = None,
                               precision_floor_ratio: float = 0.01) -> tuple[np.ndarray, Dict[str, np.ndarray | float]]:
    """EB-moderated WLS scores of a centred matrix plus the reference's details dict (inference.py:231-299)."""
    c = np.asarray(centered_matrix, dtype=np.float64)
    if c.ndim != 2:
        raise ValueError("`centered_matrix` must be two-dimensional")
    if 0 in c.shape:
        raise ValueError("`centered_matrix` must be non-empty")
    floor_ratio = float(max(precision_floor_ratio, 0.0))
    out = _wls_native.score_centered_wls(
        c, lower_bound_z=float(lower_bound_z), prior_df=float(prior_df), min_effect=min_effect,
        spatial_window=31 if spatial_window is None else int(spatial_window), precision_floor_ratio=floor_ratio)
    scores = np.asarray(out[0], dtype=np.float64)
    details: Dict[str, np.ndarray | float] = {k: np.asarray(v, dtype=np.float64) for k, v in zip(_WLS_FIELDS, out[1:6])}
    details["z_scores"] = details["mean"] / np.maximum(details["standard_error"], 1.0e-8)
    _finite_or_raise("EB scoring produced non-finite values", scores, *(details[k] for k in _WLS_FIELDS), details["z_scores"])
    details.update(min_effect=float(0.0 if min_effect is None else max(min_effect, 0.0)), precision_floor_ratio=floor_ratio,
                   degrees_of_freedom=np.full(c.shape[1], float(out[6]), dtype=np.float64), prior_spatial_window=float(out[7]))
    return scores, details


def score_loci_wls(chrom_matrix: np.ndarray, lower_bound_z: float = 1.0, prior_df: float = 5.0,
                   min_effect: float | None = None, precision_floor_ratio: float = 0.01, low_memory: bool = False,
                   return_details: bool = False) -> np.ndarray | Tuple[np.ndarray, Dict[str, Any]]:
    r"""Score loci with an EB-moderated summary on baseline-corrected log signal (inference.py:302-379).

    float32 input is uploaded as float32 (half the host->device bytes) and widened on the device,
    which is exactly ``np.asarray(chrom_matrix, dtype=np.float64)`` of the reference."""
    matrix_in = np.asarray(chrom_matrix)
    if matrix_in.dtype != np.float32:
        matrix_in = np.asarray(matrix_in, dtype=np.float64)
    if matrix_in.ndim != 2:
        if np.any(~np.isfinite(matrix_in)):
            raise ValueError("`chrom_matrix` contains non-finite values")
        raise ValueError("`chrom_matrix` must be two-dimensional")
    if matrix_in.shape[0] == 0 or matrix_in.shape[1] == 0:
        raise ValueError("`chrom_matrix` must be non-empty")
    matrix_in = np.ascontiguousarray(matrix_in)
    m, n = matrix_in.shape
    lib = _lib.load()
    _lib.require_device()
    prm = score_params(lower_bound_z, prior_df, min_effect, precision_floor_ratio)

    names = ("scores", "mean", "raw_variance", "prior_variance", "moderated_variance", "standard_error")
    bufs = {k: np.zeros(n, dtype=np.float64) for k in (names if return_details else names[:1])}
    out = _lib.ScoreOutputs()
    for k, v in bufs.items():
        setattr(out, k, v.ctypes.data)
    centered = None
    if return_details:
        centered = np.zeros((m, n), dtype=np.float64)
        out.centered_matrix = centered.ctypes.data
    fn = lib.rocco_score_loci_wls_f32 if matrix_in.dtype == np.float32 else lib.rocco_score_loci_wls_f64
    st = fn(_lib.np_ptr(matrix_in), m, n, ctypes.byref(prm), ctypes.byref(out))
    if st == _lib.ST_NONFINITE:
        if np.any(~np.isfinite(matrix_in)):
            raise ValueError("`chrom_matrix` contains non-finite values")
        raise ValueError("Locus scoring produced non-finite values")
    _lib.check(st, "score_loci_wls")
    scores = bufs["scores"]
    if not return_details:
        return scores.astype(np.float64)
    se = bufs["standard_error"]
    details = {
        "input_scale": "log2p1",
        "local_baseline_window": int(out.baseline_window),
        "local_baseline_lambda": float(out.baseline_lambda),
        "mean": bufs["mean"],
        "raw_variance": bufs["raw_variance"],
        "prior_variance": bufs["prior_variance"],
        "moderated_variance": bufs["moderated_variance"],
        "standard_error": se,
        "z_scores": bufs["mean"] / np.maximum(se, 1.0e-8),
        "min_effect": float(0.0 if min_effect is None else max(min_effect, 0.0)),
        "precision_floor_ratio": float(max(precision_floor_ratio, 0.0)),
        "prior_spatial_window": int(out.resolved_spatial_window),
        "degrees_of_freedom": np.full(n, float(out.total_df), dtype=np.float64),
        "centered_matrix": centered.astype(np.float32 if low_memory else np.float64, copy=False),
    }
    return scores.astype(np.float64), details


# ------------------------------------------------------------------------------------------------
# Budget null: dependent wild residual bootstrap (inference.py:446-1148) -- SURVEY.md 8(f) rank 1
# ------------------------------------------------------------------------------------------------
def _resolve_budget_ess_max_lag(n_loci: int, dependence_lag_hint: int | None = None) -> int:
    r"""ESS autocorrelation lag cap (inference.py:504-517)."""
    return int(_lib.load().rocco_b200_budget_ess_max_lag(int(max(1, n_loci)), _hint(dependence_lag_hint)))


def _resolve_budget_bootstrap_bandwidth(n_loci: int, dependence_lag_hint: int | None = None) -> int:
    r"""Bartlett bandwidth of the multiplier field (inference.py:520-530)."""
    return int(_lib.load().rocco_b200_budget_bandwidth(int(max(1, n_loci)), _hint(dependence_lag_hint)))


def _hint(dependence_lag_hint) -> int:
    # the C entries use "<= 0" for "no hint"; a non-positive hint means max(8, hint) = 8 bins / 4 * max(1, hint) = 4 in the
    # reference, which the smallest positive hint reproduces
    if dependence_lag_hint is None:
        return 0
    return max(1, int(dependence_lag_hint))


def _build_budget_bootstrap_kernel(bandwidth: int) -> np.ndarray:
    r"""Bartlett taps on [-b, b] with unit L2 norm (inference.py:533-541); host helper."""
    b = int(max(1, bandwidth))
    taps = np.maximum(1.0 - np.abs(np.arange(-b, b + 1, dtype=np.float64)) / float(b + 1), 0.0)
    return taps / np.sqrt(np.sum(taps * taps))


def _estimate_effective_sample_size(values: np.ndarray, max_lag: int) -> tuple[float, float, int]:
    r"""ESS from the integrated autocorrelation time with Geyer's truncation (inference.py:446-501); the
    autocovariances are direct lag products on the device instead of an FFT."""
    values_ = np.ascontiguousarray(values, dtype=np.float64)
    if values_.ndim != 1:
        raise ValueError("`values` must be one-dimensional")
    n_eff, tau, used = ctypes.c_double(), ctypes.c_double(), ctypes.c_int()
    if values_.size >= 4:
        _lib.require_device()
    st = _lib.load().rocco_effective_sample_size_f64(_lib.np_ptr(values_), values_.size, int(max_lag), ctypes.byref(n_eff),
                                                     ctypes.byref(tau), ctypes.byref(used))
    if st == _lib.ST_NONFINITE:                       # non-finite series: the reference returns (n, 1, 0) (inference.py:470-471)
        return float(values_.size), 1.0, 0
    _lib.check(st, "effective sample size")
    return float(n_eff.value), float(tau.value), int(used.value)


RANDOM_STREAMS = {"philox": 0, "numpy": 1}


def random_streams_code(random_streams: str, random_seed, innovations) -> int:
    """The native code of a ``random_streams`` choice of the budget null, after checking it.

    ``"philox"`` (the default): counter-based Philox4x32-10 streams keyed by ``random_seed``; the null agrees with the
    reference in distribution.  ``"numpy"``: the reference's own streams -- draw d takes its normals from
    ``numpy.random.default_rng(random_seed + 104729 * (d + 1))``, the samples served in order -- generated on the device,
    so the null is the reference's.  ``"numpy"`` needs ``0 <= random_seed < 2**64`` (NumPy rejects negative seeds) and
    excludes ``innovations``, which replace the generator."""
    if random_streams not in RANDOM_STREAMS:
        raise ValueError(f"`random_streams` must be one of {sorted(RANDOM_STREAMS)}, got {random_streams!r}")
    if random_streams == "numpy":
        if innovations is not None:
            raise ValueError("`random_streams='numpy'` generates the innovations: do not pass `innovations` as well")
        if int(random_seed) < 0:
            raise ValueError("`random_seed` must be non-negative with `random_streams='numpy'` (as for numpy.random.default_rng)")
        if int(random_seed) >= 1 << 64:
            raise ValueError("`random_seed` must be below 2**64")
    return RANDOM_STREAMS[random_streams]


def budget_params(score, dependence_lag_hint=None, num_null_draws=25, min_null_draws=None, stability_abs_tol=5.0e-3,
                  stability_rel_tol=5.0e-2, random_seed=0, random_streams="philox", sample_offset=0, d_innovations=None):
    """The native parameters of the budget null: the ``ScoreParams`` ``score`` and the null's settings, as the estimator
    entries take them.  ``sample_offset``: global index of this rank's first sample (sample sharding); ``d_innovations``:
    a CUDA tensor of supplied innovations, or None.  Raises ``ValueError`` as ``random_streams_code``."""
    prm = _lib.BudgetParams()
    _lib.load().rocco_b200_default_budget_params(ctypes.byref(prm))
    prm.score = score
    prm.dependence_lag_hint = _hint(dependence_lag_hint)
    prm.num_null_draws = int(max(1, num_null_draws))
    prm.min_null_draws = 0 if min_null_draws is None else int(max(1, min_null_draws))
    prm.stability_abs_tol = float(stability_abs_tol)
    prm.stability_rel_tol = float(stability_rel_tol)
    prm.random_seed = int(random_seed) & 0xFFFFFFFFFFFFFFFF
    prm.random_streams = random_streams_code(random_streams, random_seed, d_innovations)
    prm.sample_offset = int(sample_offset)
    prm.d_innovations = None if d_innovations is None else d_innovations.data_ptr()
    return prm


def _budget_details(res: "_lib.BudgetResult") -> Dict[str, Any]:
    d = {k: float(getattr(res, k)) for k in (
        "observed_positive_fraction", "observed_negative_fraction", "null_positive_fraction", "observed_excess_mass",
        "observed_excess_units", "null_threshold", "observed_tail_occupancy", "null_tail_occupancy",
        "null_tail_occupancy_sd", "null_tail_occupancy_stderr", "null_center", "null_scale", "nonnull_fraction",
        "effective_count", "effective_total_count", "autocorrelation_time", "negative_fraction",
        "null_reference_mean_positive_consensus", "null_reference_max_positive_consensus")}
    d.update({
        "null_excess_mass": float(res.null_positive_mass), "null_excess_units": float(res.null_positive_units),
        "null_excess_units_sd": float(res.null_positive_units_sd),
        "null_excess_units_stderr": float(res.null_positive_units_stderr),
        "ess_max_lag": float(res.ess_max_lag), "ess_lags_used": float(res.ess_lags_used), "num_loci": float(res.num_loci),
        "negative_support_size": float(res.negative_support_size), "num_null_draws": float(res.num_null_draws),
        "max_null_draws": float(res.max_null_draws), "adaptive_stop": bool(res.adaptive_stop),
        "wild_bandwidth": float(res.wild_bandwidth), "wild_process": "bartlett_multiplier",
        "null_method": "dependent_wild_residual_bootstrap",
        # not in the reference's dict: inputs of rocco._resolve_chrom_gamma, computed while the scores are on the device
        "positive_score_median": float(res.positive_score_median), "positive_score_count": int(res.positive_score_count),
    })
    return d


def estimate_budget_nonnull_fraction_from_wild_bootstrap_null(
        centered_matrix: np.ndarray, observed_scores: np.ndarray | None = None, lower_bound_z: float = 1.0,
        prior_df: float = 5.0, min_effect: float | None = None, precision_floor_ratio: float = 0.01,
        dependence_lag_hint: int | None = None, num_null_draws: int = 25, random_seed: int = 0,
        progress_label: str | None = None, num_processes: int = 1, return_details: bool = False,
        min_null_draws: int | None = None, stability_abs_tol: float = 5.0e-3, stability_rel_tol: float = 5.0e-2,
        innovations: np.ndarray | None = None, random_streams: str = "philox") -> float | Tuple[float, Dict[str, Any]]:
    r"""Conservative enriched fraction from a dependent-wild-bootstrap null (inference.py:988-1148).

    Same arguments, return value and details keys as the reference.  The whole estimator -- null template, fitted-null
    score field, up to ``num_null_draws`` multiplier fields each re-scored by the WLS chain, the adaptive stop, the
    observed-side summary and the ESS -- runs on the GPU in one native call; ``num_processes`` and ``progress_label``
    are accepted and unused.  ``random_streams="philox"`` (the default) draws Philox streams keyed by ``random_seed``:
    results agree with the reference in distribution.  ``random_streams="numpy"`` generates the reference's own NumPy
    PCG64 streams on the device, so the draws, and the result, are the reference's (see ``random_streams_code``).
    ``innovations`` (``[num_null_draws, n_samples, n_loci + 2*bandwidth]`` iid N(0,1)) replaces the generator, e.g. to
    replay the reference's own streams from the host.
    """
    random_streams_code(random_streams, random_seed, innovations)     # budget_params does not see host innovations
    centered = np.asarray(centered_matrix, dtype=np.float64)
    if centered.ndim == 1:
        centered = centered[np.newaxis, :]
    if centered.ndim != 2:
        raise ValueError("`centered_matrix` must be one- or two-dimensional")
    m, n = centered.shape
    if n <= 0:
        raise ValueError("`centered_matrix` must contain at least one locus")
    if m == 0:
        raise ValueError("`centered_matrix` must be non-empty")
    centered = np.ascontiguousarray(centered)
    obs = None
    if observed_scores is not None:
        obs = np.ascontiguousarray(observed_scores, dtype=np.float64)
        if obs.shape[0] != n:
            raise ValueError("`observed_scores` must have the same number of loci as `centered_matrix`")
    lib = _lib.load()
    _lib.require_device()
    prm = budget_params(score_params(lower_bound_z, prior_df, min_effect, precision_floor_ratio), dependence_lag_hint,
                        num_null_draws, min_null_draws, stability_abs_tol, stability_rel_tol, random_seed, random_streams)
    inn = None
    if innovations is not None:
        bw = _resolve_budget_bootstrap_bandwidth(n, dependence_lag_hint)
        inn = np.ascontiguousarray(innovations, dtype=np.float64)
        if inn.shape != (prm.num_null_draws, m, n + 2 * bw):
            raise ValueError(f"`innovations` must have shape {(prm.num_null_draws, m, n + 2 * bw)}")
    res = _lib.BudgetResult()
    st = lib.rocco_budget_nonnull_fraction_f64(_lib.np_ptr(centered), m, n, None if obs is None else _lib.np_ptr(obs),
                                               ctypes.byref(prm), None if inn is None else _lib.np_ptr(inn), ctypes.byref(res))
    if st == _lib.ST_NONFINITE:
        raise ValueError("Budget initialization produced non-finite values")
    _lib.check(st, "budget null")
    details = _budget_details(res)
    if return_details:
        return float(res.nonnull_fraction), details
    return float(res.nonnull_fraction)


def estimate_budget_nonnull_fraction_from_empirical_null(centered_matrix, observed_scores=None, lower_bound_z=1.0, prior_df=5.0,
                                                         min_effect=None, precision_floor_ratio=0.01, dependence_lag_hint=None,
                                                         num_null_draws=25, random_seed=0, progress_label=None,
                                                         num_processes=1, return_details=False):
    r"""Wrapper for the wild-bootstrap budget estimator (inference.py:1424-1452)."""
    return estimate_budget_nonnull_fraction_from_wild_bootstrap_null(
        centered_matrix, observed_scores=observed_scores, lower_bound_z=lower_bound_z, prior_df=prior_df,
        min_effect=min_effect, precision_floor_ratio=precision_floor_ratio, dependence_lag_hint=dependence_lag_hint,
        num_null_draws=num_null_draws, random_seed=random_seed, progress_label=progress_label,
        num_processes=num_processes, return_details=return_details)


# ------------------------------------------------------------------------------------------------
# empirical-Bayes chromosome budgets (inference.py:1488-1737) -- SURVEY.md 8(f) rank 2
#
# Twenty-four numbers per genome: this stays on the host with SciPy exactly as in the reference (the
# optimiser's iterates decide the last digits, so the same optimiser is used on the same objective).
# ------------------------------------------------------------------------------------------------
def _raw_rate_summary(successes: np.ndarray, totals: np.ndarray) -> tuple[float, float, float]:
    """(pooled rate clipped to [1e-6, 1 - 1e-6], sample variance of the raw rates, binomial floor of that variance)"""
    trials = np.maximum(totals, 1.0)
    rates = successes / trials
    pooled = float(np.clip(np.sum(successes) / max(np.sum(totals), 1.0), 1.0e-6, 1.0 - 1.0e-6))
    spread = float(np.var(rates, ddof=1)) if rates.size > 1 else 0.0
    floor = float(pooled * (1.0 - pooled) * np.mean(1.0 / trials))
    return pooled, spread, floor


def fit_beta_prior_mle(successes: np.ndarray, totals: np.ndarray, init_center: float = 0.05,
                       init_strength: float = 10.0) -> Tuple[float, float]:
    r"""Maximum-likelihood (alpha, beta) of a beta-binomial over chromosomes, L-BFGS-B on (log alpha, log beta).

    When the raw rates are no more dispersed than binomial sampling alone explains, the fit sits on the boundary
    rho = 0 and a (practically) infinitely strong prior at the pooled rate is returned (inference.py:1520-1528)."""
    from scipy import optimize, special
    x = np.asarray(successes, dtype=np.float64)
    n = np.asarray(totals, dtype=np.float64)
    if x.shape != n.shape:
        raise ValueError("`successes` and `totals` must have the same shape")
    if x.size == 0:
        return 1.0, 1.0
    center = min(max(float(init_center), 1.0e-6), 1.0 - 1.0e-6)
    pooled, spread, floor = _raw_rate_summary(x, n)
    if spread <= floor + 1.0e-12:
        strength = float(max(1.0e12, 100.0 * np.max(n)))
        return pooled * strength, (1.0 - pooled) * strength
    weak = (center * float(init_strength), (1.0 - center) * float(init_strength))

    def negative_loglik(theta: np.ndarray) -> float:
        a, b = float(np.exp(theta[0])), float(np.exp(theta[1]))
        return float(-np.sum(special.betaln(x + a, n - x + b) - special.betaln(a, b)))

    fit = optimize.minimize(negative_loglik, np.log(np.array(weak, dtype=np.float64)), method="L-BFGS-B")
    if not fit.success:
        logger.warning("Falling back to a weak beta prior while fitting EB budgets: %s", fit.message)
        return weak
    return float(np.exp(fit.x[0])), float(np.exp(fit.x[1]))


def _beta_posterior_budget_quantile(successes: float, total: float, alpha: float, beta: float, posterior_quantile: float,
                                    min_budget: float, max_budget: float) -> float:
    from scipy import stats
    a = float(max(1.0e-12, successes + alpha))
    b = float(max(1.0e-12, (total - successes) + beta))
    q = float(np.clip(posterior_quantile, 1.0e-6, 1.0 - 1.0e-6))
    return float(np.clip(float(stats.beta.ppf(q, a, b)), min_budget, max_budget))


def estimate_empirical_bayes_budgets(chrom_candidate_counts: Dict[str, float], chrom_total_counts: Dict[str, float],
                                     min_budget: float = 1.0e-4, max_budget: float = 0.5, init_center: float = 0.05,
                                     init_strength: float = 10.0, posterior_quantile: float = 0.01
                                     ) -> Tuple[Dict[str, float], Dict[str, float]]:
    r"""Per-chromosome budgets shrunk towards a genome-wide beta prior (inference.py:1593-1737).

    One chromosome: the default prior (init_center, init_strength); two or three: a weak prior at the pooled rate;
    more: the beta-binomial MLE.  The budget is a LOW quantile of each chromosome's beta posterior, clipped to
    [min_budget, max_budget].  Returns (budgets, meta) with the reference's meta keys."""
    chroms = list(chrom_candidate_counts.keys())
    if chroms != list(chrom_total_counts.keys()):
        raise ValueError("`chrom_candidate_counts` and `chrom_total_counts` must share keys in the same order")
    x = np.array([chrom_candidate_counts[c] for c in chroms], dtype=np.float64)
    n = np.array([chrom_total_counts[c] for c in chroms], dtype=np.float64)
    pooled, spread, floor = _raw_rate_summary(x, n)
    q = float(posterior_quantile)
    if not (0.0 < q < 1.0):
        raise ValueError("`posterior_quantile` must lie strictly between 0 and 1")
    at_floor = bool(spread <= floor + 1.0e-12)
    if len(chroms) <= 1:
        alpha, beta = float(init_center) * float(init_strength), (1.0 - float(init_center)) * float(init_strength)
        centre, strength, method, flag = float(init_center), float(init_strength), "single_chrom_default", False
        dispersion = 1.0 / (1.0 + alpha + beta)
    elif len(chroms) <= 3:
        alpha, beta = pooled * float(init_strength), (1.0 - pooled) * float(init_strength)
        centre, strength, method, flag = pooled, float(alpha + beta), "weak_pooled_prior", at_floor
        dispersion = max(0.0, 1.0 / (1.0 + strength))
    else:
        alpha, beta = fit_beta_prior_mle(x, n, init_center=init_center, init_strength=init_strength)
        centre, strength, method, flag = float(alpha / (alpha + beta)), float(alpha + beta), "beta_binomial_mle", at_floor
        dispersion = max(0.0, 1.0 / (1.0 + strength))
    budgets = {c: _beta_posterior_budget_quantile(x[k], n[k], alpha, beta, q, min_budget, max_budget) for k, c in enumerate(chroms)}
    meta = {
        "alpha": float(alpha), "beta": float(beta), "genome_wide_budget": float(centre), "prior_strength": float(strength),
        "prior_dispersion": float(dispersion), "min_prior_dispersion": 0.0, "observed_raw_budget_var": float(spread),
        "theoretical_min_raw_budget_var": float(floor), "prior_dispersion_at_floor": bool(flag),
        "posterior_summary": "beta_quantile", "posterior_quantile": float(q), "prior_fit_method": method,
    }
    return budgets, meta
