/*
 * rocco_b200 -- C-ABI of the B200-native consensus-selection hot path.
 *
 * This is the drop-in boundary for ROCCO's three hot-path extensions (SURVEY.md section 8b):
 *
 *   reference interface (under /root/reference/rocco)            replaced by
 *   -----------------------------------------------------------  -----------------------------------------
 *   native/baseline_backend.h:11-22                               rocco_crossfit_whittaker_baseline_f64
 *     rocco_crossfit_whittaker_baseline_f64 / _matrix_f64         rocco_crossfit_whittaker_baseline_matrix_f64
 *   native/wls_backend.h:11-28  rocco_score_centered_wls_f64      rocco_score_centered_wls_f64
 *   _chain_dp.c:9-213 (kernel inline in the CPython wrapper;      rocco_solve_penalized_chain_f64
 *     no C-ABI upstream)
 *   dp.py:89-164  calibrate_selection_penalty (62 DP passes       rocco_calibrate_selection_penalty_f64
 *     driven from Python)
 *   inference.py:302-379 score_loci_wls (log2p1 -> row median     rocco_score_loci_wls_f64 / _f32
 *     -> baseline -> centered WLS, four m x n temporaries)
 *   rocco.py:243-355 column statistics over the sample axis       rocco_column_stat_f64
 *   rocco.py:139-191 mask -> merged intervals                     rocco_mask_to_intervals_u8
 *
 * The first three keep the reference's exact symbol names, argument order and status codes and
 * take HOST pointers, so the reference's own CPython wrappers (_baseline.c, _wls.c) link against
 * librocco_b200.so unchanged (INTEGRATION.md).  Everything is plain pointers and sizes; there are
 * no torch types here.  The `*_dev` entry points take DEVICE pointers and a CUDA stream so the
 * stages chain on the GPU without host round trips; they are what the Python host side and the
 * benchmark use.
 *
 * Status codes (reference: wls_backend.c:779-788, _wls.c:133-150, _baseline.c:96-101):
 *    0  ok        -1  allocation failure (-> MemoryError)      -2  invalid input (-> ValueError)
 *   -3  CUDA runtime error (-> RuntimeError; text from rocco_b200_last_error())
 *   -4  non-finite values in the input / result (-> ValueError, inference.py:45,207,289-298)
 * There is NO CPU fallback: without a CUDA device every compute entry returns -3.
 */
#ifndef ROCCO_B200_H
#define ROCCO_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* ------------------------------------------------------------------ library / device */
const char *rocco_b200_version(void);
const char *rocco_b200_last_error(void);          /* thread-local text of the last -3 */
int rocco_b200_device_count(void);                /* 0 when no CUDA device is visible */
int rocco_b200_set_device(int device);
/* Number of kernels this library has launched in this process (bench.py's gpu_launches). */
unsigned long long rocco_b200_kernel_launches(void);
/* Return the scratch the library's stream-ordered memory pools are holding beyond `bytes_to_keep` (per pool) to the
 * driver, so that other allocators in the process (torch's, a second workload) can use it.  Returns pools trimmed. */
int rocco_b200_trim_pools(size_t bytes_to_keep);

/* Per-kernel timing with CUDA events on the launching stream (off by default).  report() synchronises,
 * writes "<scope> <total_ms> <launch_sets> <algorithmic_bytes>" lines into buf and clears the log. */
int rocco_b200_profile_enable(int on);
int rocco_b200_profile_report(char *buf, size_t capacity);
/* "<scope> <start_ms> <duration_ms>" per recorded scope in record order (start relative to the first scope); keeps the log. */
int rocco_b200_profile_timeline(char *buf, size_t capacity);

/* ------------------------------------------------------------------ reference-named host entries */
int rocco_crossfit_whittaker_baseline_f64(
    const double *y_values, size_t value_count, double penalty_lambda, double *baseline_out);
int rocco_crossfit_whittaker_baseline_matrix_f64(
    const double *matrix_values, size_t row_count, size_t column_count,
    double penalty_lambda, double *baseline_out);
int rocco_score_centered_wls_f64(
    const double *centered_matrix, size_t sample_count, size_t locus_count,
    double lower_bound_z, double prior_df, double min_effect, int use_min_effect,
    int spatial_window, double precision_floor_ratio,
    double *mean_out, double *raw_variance_out, double *prior_variance_out,
    double *moderated_variance_out, double *standard_error_out, double *scores_out,
    double *degrees_of_freedom_out, int *resolved_window_out);

/* ------------------------------------------------------------------ chain DP + multiplier search */
typedef struct rocco_b200_chain_result {
    double selection_penalty;     /* lambda the mask was solved at                              */
    double penalized_objective;   /* sum (s-lambda) z - sum c |dz|   (reference: DP best value)  */
    double objective;             /* -sum s z + sum c |dz|           (dp.py:16-34)               */
    long long selected_count;     /* sum z                                                       */
    long long switch_count;       /* number of 0/1 boundaries in the mask                        */
    long long exact_tie_bins;     /* decisions that needed the (value, fewer-count) tie-break    */
    long long near_tie_bins;      /* decisions within 1e-9*(1+|c|) of a threshold (documented)   */
    int dp_passes;                /* DP passes the reference spends on this search (62 by default) */
    int search_rounds;            /* batched launch sets actually used (each evaluates 2^L-1 multipliers) */
    int status;                   /* 0, or -2 / -4 for this chromosome                           */
    int reserved;
} rocco_b200_chain_result;

/* One DP solve at a fixed multiplier.  `switch_costs` has length n-1 (may be NULL when n == 1).
 * Replaces _chain_dp.solve_penalized_chain(scores, switch_costs, selection_penalty).           */
int rocco_solve_penalized_chain_f64(
    const double *scores, const double *switch_costs, size_t n, double selection_penalty,
    uint8_t *solution_out, double *penalized_objective_out, long long *selected_count_out);

/* dp.py:89-164: bracket + `max_iter` dyadic bisection steps; returns the upper end and its mask. */
int rocco_calibrate_selection_penalty_f64(
    const double *scores, const double *switch_costs, size_t n, long long target_count,
    int max_iter, double *selection_penalty_out, uint8_t *solution_out,
    double *penalized_objective_out, long long *selected_count_out);

/* Device-resident, many chromosomes per call.  Chromosome c owns scores[offset_c .. offset_c+n_c).
 * mode: 0 = fixed multiplier `selection_penalty`, 1 = budget search to `target_count`.
 * `cost_sum` is sum(switch_costs) as the caller's host library computes it (dp.py:110-111 uses
 * numpy.sum, whose rounding defines the bracket); gamma is the constant switch cost
 * (dp.py:37-46).  d_switch_costs, when not NULL, is a per-bin cost vector laid out like scores
 * (entry i = cost between bins i and i+1 of that chromosome; the last entry of each is unused). */
typedef struct rocco_b200_chain_task {
    size_t offset;
    size_t n;
    double gamma;
    double cost_sum;
    double selection_penalty;
    long long target_count;
    int mode;
    int max_iter;
} rocco_b200_chain_task;

int rocco_b200_chain_solve_batch_dev(
    const double *d_scores, const double *d_switch_costs,
    const rocco_b200_chain_task *tasks, int task_count,
    uint8_t *d_masks_out,                 /* same layout as d_scores, one byte per bin */
    rocco_b200_chain_result *results_out, /* host, task_count entries                   */
    int levels_per_round,                 /* bisection levels evaluated per launch (1..8); 0 = default */
    void *cuda_stream);

/* Genome-wide budget (opt-in; not a behaviour of the reference, which searches one multiplier per chromosome, dp.py:197-207):
 * ONE multiplier for a genome spread over this call's chromosomes and those of every other rank that takes part.  The
 * search is dp.py:89-164 applied to the concatenated chain S = s_1 || s_2 || ... with switch costs c_1 || 0 || c_2 || 0 ...
 * (a zero cost at each junction decouples the chromosomes, so its mask at any multiplier is the per-chromosome masks laid
 * end to end): target = floor(N * budget) over N = sum n_c, bracket min(S) - cost_sum - 1 .. max(S) + cost_sum + 1, then
 * `max_iter` bisection levels on the genome's count; every chromosome is solved at the returned upper end.  All fields
 * are agreed by the ranks before the call (like the shapes of the sharded budget null).  cost_sum is the correctly rounded
 * sum of the genome's switch costs, so it does not depend on how chromosomes are ordered or spread over ranks. */
typedef struct rocco_b200_genome_search {
    long long total_bins;        /* N over all ranks                                                           */
    long long target_count;      /* floor(N * budget)                                                          */
    double cost_sum;             /* correctly rounded sum of every switch cost                                 */
    double cost_max;             /* largest switch cost of the genome                                          */
    double score_min, score_max; /* genome extremes; NaN: from this call's chromosomes (valid only without a reducer) */
    int max_iter;
    int reserved;
} rocco_b200_genome_search;

typedef struct rocco_b200_genome_result {
    double selection_penalty;    /* the genome's multiplier (0.0 when target >= N)                              */
    long long selected_count;    /* selected bins of the whole genome                                          */
    int dp_passes;               /* DP passes the reference's search would spend (62 by default)                */
    int search_rounds;           /* batched launch sets, each followed by one reduce                           */
    int status;
    int reserved;
} rocco_b200_genome_result;

/* `tasks` as for rocco_b200_chain_solve_batch_dev; their mode, target_count and selection_penalty are ignored.  task_count
 * may be 0 on a rank that holds no chromosome (it still takes part in every reduce).  `allreduce` (rocco_b200_allreduce_fn,
 * below; NULL when this call holds the whole genome) is called once per search round on 2^L + 1 doubles, L the largest tree
 * depth (levels_per_round, which every rank passes alike): the counts of the round's multipliers summed over this rank's
 * chromosomes, its live-tile count and a status slot; every rank then takes the same decision on the same integers.  One
 * last reduce sums the selected counts of the final masks.  A rank-local failure after the first allocation (the reduce
 * buffer) is carried to the next reduce, and every rank returns that status.  Argument errors are returned at once:
 * check them across ranks first.  Exact search (rocco_b200_chain_set_exact_search) is rejected with -2. */
int rocco_b200_chain_solve_genome_dev(
    const double *d_scores, const double *d_switch_costs,
    const rocco_b200_chain_task *tasks, int task_count,
    const rocco_b200_genome_search *search,
    int (*allreduce)(double *d_buf, size_t count, void *cuda_stream, void *user), void *user,
    uint8_t *d_masks_out, rocco_b200_chain_result *results_out, rocco_b200_genome_result *genome_out,
    int levels_per_round, void *cuda_stream);

/* Chromosomes of at most `max_bins` (<= 4096, the default) bins are solved by replaying the
 * reference's sequential recurrence operation for operation (bit-identical value / count / mask);
 * longer ones use the parallel scan.  Returns the previous setting.  0 forces the scan everywhere. */
int rocco_b200_chain_set_seq_max(int max_bins);
/* Exact search (off by default): every multiplier at which some decision lies within 1e-7 (1 + c) of its threshold -- i.e.
 * inside the rounding noise of the reference's absolute-value recurrence, which is where the last bisection levels land --
 * is re-evaluated by replaying that recurrence sequentially over the whole chromosome (_chain_dp.c:109-186).  The
 * returned multiplier and mask are then the reference's bits for ANY length, at ~13 ns per bin per replayed pass.
 * Returns the previous setting. */
int rocco_b200_chain_set_exact_search(int on);
/* Search rounds skip tiles whose decisions provably cannot change inside the remaining bracket (default on; 0 evaluates every
 * tile in every round -- same counts, used for A/B checks).  Returns the previous setting. */
int rocco_b200_chain_set_tile_freezing(int on);

/* Multiplier sweep: counts and objectives for `lambda_count` multipliers in one launch set
 * (BASELINE.json config 5).  Outputs are host arrays of lambda_count entries. */
int rocco_b200_chain_sweep_dev(
    const double *d_scores, size_t n, double gamma,
    const double *lambdas, int lambda_count,
    long long *selected_count_out, double *penalized_objective_out, double *objective_out,
    void *cuda_stream);

/* ------------------------------------------------------------------ mask -> merged intervals */
/* rocco.py:179-191 + 74-95: bins with mask > 0, the LAST bin dropped, adjacent bins merged,
 * runs shorter than min_length_bp removed.  Emits (start, end) = (first + i*step, first + j*step).
 * Returns the number of intervals (>= 0) or a negative status; capacity is in intervals. */
long long rocco_mask_to_intervals_u8(
    const uint8_t *mask, size_t n, long long first_start, long long step, long long min_length_bp,
    long long *starts_out, long long *ends_out, size_t capacity);
long long rocco_b200_mask_to_intervals_dev(
    const uint8_t *d_mask, size_t n, long long first_start, long long step, long long min_length_bp,
    long long *starts_out, long long *ends_out, size_t capacity, void *cuda_stream);

/* Batched form: chromosome c occupies mask[offsets[c] .. offsets[c]+lengths[c]) (ascending, disjoint,
 * padding bytes zero).  One pass over the concatenated masks; outputs are bin indices relative to
 * each chromosome (end exclusive) plus the chromosome index of every run. */
long long rocco_b200_mask_to_runs_batch_dev(
    const uint8_t *d_mask, const size_t *offsets, const size_t *lengths, int chrom_count,
    long long *start_bin_out, long long *end_bin_out, int *chrom_index_out, size_t capacity,
    void *cuda_stream);

/* narrowPeak summit offsets (rocco.py:840-872, SURVEY.md 8(f) rank 4): for peak p = [peak_starts[p], peak_ends[p]) the bins
 * whose start lies inside it are searched for the largest mean (float32 track as the reference stores it; NaN ignored,
 * first occurrence wins, at least one finite value required); offsets_out[p] = clip(centre of that bin - start, 0, len-1),
 * or -1 when the peak is empty, has non-positive length or no finite mean.  track_starts must be ascending. */
int rocco_narrowpeak_summit_offsets_f32(const long long *track_starts, const long long *track_centers, const float *track_mean,
                                        size_t n_track, const long long *peak_starts, const long long *peak_ends,
                                        size_t n_peaks, long long *offsets_out);
int rocco_b200_summit_offsets_dev(const long long *d_track_starts, const long long *d_track_centers, const float *d_track_mean,
                                  size_t n_track, const long long *d_peak_starts, const long long *d_peak_ends,
                                  size_t n_peaks, long long *d_offsets_out, void *cuda_stream);

/* numpy.sum of a float64 vector / of n copies of one value, restated bit-exactly (host helpers:
 * dp.py:110-111 builds the search bracket from numpy.sum(switch_costs)). */
/* Host helper: write n BED3 records (BED4 with chrom_start_end names when name_features != 0) to `path`
 * (rocco.py:98-110 _write_bed_records).  Record i uses names[name_idx[i]] (name_idx == NULL: names[0]). */
int rocco_b200_write_bed3(const char *path, const char *const *names, int n_names, const int *name_idx,
                          const long long *starts, const long long *ends, size_t n, int name_features);
/* The same text written into `path` at byte `offset` without truncating the file (created if missing): processes that
 * know each other's text sizes assemble ONE BED file without a gather pass (the multi-rank form of rocco.py:194-240's
 * output).  *bytes_written (may be NULL) returns the size of the text. */
int rocco_b200_write_bed3_at(const char *path, long long offset, const char *const *names, int n_names, const int *name_idx,
                             const long long *starts, const long long *ends, size_t n, int name_features,
                             long long *bytes_written);
/* Host helper: combine_chrom_results (rocco.py:194-240) over canonical BED text -- read `n_paths` files, order the
 * records by (chrom, start, end), merge overlapping/abutting records per chrom, write BED3 (BED4 when name_features).
 * Returns the number of records written, or -1 when a file is not canonical BED (the caller falls back to the
 * reference-faithful line reader); *saw_extra_columns = 1 when any row had more than three fields. */
long long rocco_b200_combine_bed3(const char *const *paths, int n_paths, const char *out_path, int name_features,
                                  int *saw_extra_columns);
/* Upload `bytes` from PINNED host memory with a kernel that reads it over PCIe (no DMA command): small uploads are then
 * not queued behind the bulk count-matrix copies other host threads have submitted.  Stream-ordered, asynchronous. */
int rocco_b200_pull_pinned(void *d_dst, const void *h_pinned, size_t bytes, void *cuda_stream);
int rocco_b200_uniform_step_i64(const long long *values, size_t n);   /* 1 iff all consecutive differences are equal */
double rocco_b200_numpy_sum_f64(const double *values, size_t n);
double rocco_b200_numpy_sum_const_f64(double value, size_t n);

/* ------------------------------------------------------------------ scoring */
typedef struct rocco_b200_score_params {
    double lower_bound_z;           /* inference.py:304 default 1.0                 */
    double prior_df;                /* 5.0 (function default) / 6.0 (CLI default)   */
    double min_effect;
    int use_min_effect;
    int spatial_window;             /* 31                                           */
    double precision_floor_ratio;   /* 0.01                                         */
    int baseline_window;            /* 101 (inference.py:185-228)                   */
    int pilot_mode;                 /* row-median pilot offset (inference.py:333): 0 = exact for n <= 4096, median of a
                                       4096-point sample above (the offset cancels in y - baseline(y): DESIGN.md section 4);
                                       1 = exact np.median for any n (one radix sort per row; validation mode)            */
} rocco_b200_score_params;

void rocco_b200_default_score_params(rocco_b200_score_params *p);

/* Order statistics of the variance trend: 0 = histogram multi-select with a sort fallback for rows whose
 * buckets overflow (default), 1 = sort every row.  Any other value means 0.  Both are exact; returns the
 * previous mode. */
int rocco_b200_trend_set_mode(int mode);
long long rocco_b200_trend_fallback_rows(void);   /* rows that took the sort path since load */
void rocco_b200_trend_fallback_reasons(long long *out8);   /* per-reason counts (diagnostics) */
long long rocco_b200_whittaker_exact_rows(void);   /* baseline rows solved by the exact sequential path since load */

/* Optional per-locus detail outputs (device or host according to the entry point); any may be NULL. */
typedef struct rocco_b200_score_outputs {
    double *scores;
    double *mean;
    double *raw_variance;
    double *prior_variance;
    double *moderated_variance;
    double *standard_error;
    double *centered_matrix;        /* m x n, optional                               */
    double total_df;                /* out */
    int resolved_spatial_window;    /* out */
    int baseline_window;            /* out */
    double baseline_lambda;         /* out */
} rocco_b200_score_outputs;

/* Full score_loci_wls on host buffers (H2D / D2H inside). matrix is row-major [sample, locus]. */
int rocco_score_loci_wls_f64(const double *matrix, size_t m, size_t n,
                             const rocco_b200_score_params *params, rocco_b200_score_outputs *out);
int rocco_score_loci_wls_f32(const float *matrix, size_t m, size_t n,
                             const rocco_b200_score_params *params, rocco_b200_score_outputs *out);

/* Device-resident variants; dtype: 0 = float64 input, 1 = float32 input. Output pointers are device. */
int rocco_b200_score_loci_wls_dev(const void *d_matrix, int dtype, size_t m, size_t n,
                                  const rocco_b200_score_params *params,
                                  rocco_b200_score_outputs *out, void *cuda_stream);
/* Sample-sharded scoring (SURVEY.md section 8e(2), BASELINE.json config 5): each rank runs the per-sample stages on
 * its own rows and writes the four per-bin sums d_acc[4][n] = {sum y/post, sum 1/post, sum 1/obs, sum 1/prior}
 * (wls_backend.c:889-911); the caller sums d_acc over ranks (one NCCL all-reduce, 32 B/bin) and finalises with
 * the TOTAL sample count (wls_backend.c:915-937). */
int rocco_b200_score_partial_dev(const void *d_matrix, int dtype, size_t m_local, size_t n,
                                 const rocco_b200_score_params *params, double *d_acc, void *cuda_stream);
/* The same, also keeping this rank's centred rows in d_centered_out [m_local][n] (device, NULL: not kept) -- the input of
 * rocco_b200_budget_nonnull_fraction_sharded_dev. */
int rocco_b200_score_partial_ex_dev(const void *d_matrix, int dtype, size_t m_local, size_t n,
                                    const rocco_b200_score_params *params, double *d_centered_out, double *d_acc,
                                    void *cuda_stream);
int rocco_b200_score_finalize_dev(const double *d_acc, size_t m_total, size_t n, const rocco_b200_score_params *params,
                                  rocco_b200_score_outputs *out, void *cuda_stream);
int rocco_b200_crossfit_baseline_dev(const double *d_rows, size_t m, size_t n, double penalty_lambda,
                                     double *d_out, void *cuda_stream);
int rocco_b200_score_centered_wls_dev(const double *d_centered, size_t m, size_t n,
                                      const rocco_b200_score_params *params,
                                      rocco_b200_score_outputs *out, void *cuda_stream);

/* ------------------------------------------------------------------ budget null (SURVEY.md 8(f) ranks 1-2)
 * Dependent-wild-bootstrap estimate of a chromosome's enriched fraction (inference.py:988-1148 on top of 446-985) and
 * the inputs of the automatic gamma (rocco.py:751-789), device-resident: fit the null residual template, score it,
 * take the null centre/scale, then re-score  template x W  for up to num_null_draws Bartlett-smoothed Gaussian
 * multiplier fields W with the reference's adaptive stop.  Innovations: Philox4x32-10 keyed by random_seed (parity with
 * the reference is statistical), or with random_streams = 1 the reference's own NumPy PCG64 streams (same normals as the
 * reference; see rocco_b200_numpy_normals_dev), unless d_innovations supplies them (bit-level replay). */
typedef struct rocco_b200_budget_params {
    rocco_b200_score_params score;  /* lower_bound_z, prior_df, min_effect, precision_floor_ratio as for the scores  */
    int dependence_lag_hint;        /* <= 0: none (bandwidth round(n^(1/3)), ESS scale 101); rocco.py:1035 passes >= 25 */
    int num_null_draws;             /* 25                                                                        */
    int min_null_draws;             /* <= 0: 8 (inference.py:795-797)                                            */
    int sample_offset;              /* global index of the first local sample (sample sharding; 0 = unsharded): row r
                                       draws the stream (Philox or NumPy) of sample sample_offset + r               */
    double stability_abs_tol;       /* 5e-3                                                                      */
    double stability_rel_tol;       /* 5e-2                                                                      */
    unsigned long long random_seed;
    const double *d_innovations;    /* optional DEVICE buffer [num_null_draws][m][n + 2*bandwidth] of iid N(0,1)
                                       (sharded: [num_null_draws][m_local][n + 2*bandwidth], this rank's rows)       */
    int random_streams;             /* innovations when d_innovations is NULL: 0 = Philox4x32-10 (default), 1 = NumPy's
                                       default_rng(random_seed + 104729 (draw + 1)).standard_normal, generated on the
                                       device, global sample i taking normals [i L, (i + 1) L), L = n + 2*bandwidth:
                                       the reference's own streams                                                   */
} rocco_b200_budget_params;

typedef struct rocco_b200_budget_result {
    double nonnull_fraction, effective_count, effective_total_count, autocorrelation_time;
    double null_center, null_scale, null_threshold;
    double null_positive_mass, null_positive_units, null_positive_fraction;
    double null_positive_units_sd, null_positive_units_stderr;
    double null_tail_occupancy, null_tail_occupancy_sd, null_tail_occupancy_stderr;
    double negative_fraction;
    double observed_positive_fraction, observed_negative_fraction, observed_excess_mass, observed_excess_units;
    double observed_tail_occupancy;
    double null_reference_mean_positive_consensus, null_reference_max_positive_consensus;
    double positive_score_median;   /* median of the observed scores > 0 (1.0 when none): rocco.py:762-769        */
    long long negative_support_size, positive_score_count, num_loci;
    int num_null_draws, max_null_draws, adaptive_stop, wild_bandwidth, ess_max_lag, ess_lags_used;
} rocco_b200_budget_result;

void rocco_b200_default_budget_params(rocco_b200_budget_params *p);
int rocco_b200_budget_bandwidth(size_t n, int dependence_lag_hint);      /* inference.py:520-530 */
int rocco_b200_budget_ess_max_lag(size_t n, int dependence_lag_hint);    /* inference.py:504-517 */
/* d_observed_scores == NULL: the scores of the fit (inference.py:752-753). */
int rocco_b200_budget_nonnull_fraction_dev(const double *d_centered, size_t m, size_t n, const double *d_observed_scores,
                                           const rocco_b200_budget_params *params, rocco_b200_budget_result *result,
                                           void *cuda_stream);
/* Sum over ranks for the sample-sharded estimator, built by the caller (NCCL is not linked into this library): replace
 * d_buf[0 .. count) (device, float64) by its sum over all ranks, in place, ordered after the work already queued on
 * `cuda_stream` and before anything queued on it later (e.g. ncclAllReduce on that stream, or a collective on a stream
 * that waits for it and that it then waits for).  Every rank calls it with the same count, the same number of times.
 * Return 0 on success; any other value aborts the call with -3 on that rank. */
typedef int (*rocco_b200_allreduce_fn)(double *d_buf, size_t count, void *cuda_stream, void *user);
/* The estimator with the SAMPLES sharded over ranks (BASELINE.json config 5): each rank passes its m_local centred rows
 * (global rows params->sample_offset .. + m_local of m_total) and the same n, observed scores and params.  The template, the
 * multiplier field and the per-row WLS stages stay local; each of the 2 + K scoring passes (fit, reference field, K draws)
 * reduces 2n column sums {sum y/post, sum 1/post} plus 4 status slots through `allreduce` (16 B/bin); everything after
 * a score track exists is recomputed by every rank from the reduced, bit-identical track, so all ranks return the same
 * result and the same status.  A rank-local failure (an allocation, a degenerate multiplier row, a non-finite local row)
 * is carried to the next reduce: every rank then returns that status; the failing rank keeps its
 * rocco_b200_last_error() text.  Not covered: a failure to allocate the 16 B/bin reduce buffer itself (the first
 * allocation of the call) and a sticky CUDA context error, after which no collective can run.  Shapes must be checked
 * across ranks before the call.  With m_local == m_total the result equals rocco_b200_budget_nonnull_fraction_dev's
 * bit for bit (allreduce may then be NULL). */
int rocco_b200_budget_nonnull_fraction_sharded_dev(const double *d_centered_local, size_t m_local, size_t n, size_t m_total,
                                                   const double *d_observed_scores, const rocco_b200_budget_params *params,
                                                   rocco_b200_allreduce_fn allreduce, void *user,
                                                   rocco_b200_budget_result *result, void *cuda_stream);
/* Building block of one draw (inference.py:653-662): d_out = d_template x W, W the Bartlett multiplier field of
 * (random_seed, draw_index), or of d_innovations [m][n + 2*bandwidth] when given.  d_out may not alias d_template. */
int rocco_b200_wild_multiply_dev(const double *d_template, size_t m, size_t n, int bandwidth,
                                 unsigned long long random_seed, unsigned draw_index, const double *d_innovations,
                                 double *d_out, void *cuda_stream);
/* Host buffers (H2D inside); `innovations` is an optional HOST buffer laid out like d_innovations. */
int rocco_budget_nonnull_fraction_f64(const double *centered, size_t m, size_t n, const double *observed_scores,
                                      const rocco_b200_budget_params *params, const double *innovations,
                                      rocco_b200_budget_result *result);
/* NumPy streams (numpy_streams.cu).  A seed is the 128-bit integer seed_hi * 2^64 + seed_lo of default_rng(seed).
 * rocco_b200_numpy_normals_dev writes normals [skip, skip + count) of default_rng(seed).standard_normal() to d_out
 * (device, count >= 1), generated on the device by a parallel parse of the ziggurat's rejection stream; words_consumed
 * (host, optional) receives how many 64-bit PCG64 outputs NumPy has drawn once it has returned normal skip + count - 1.
 * Fast-path and wedge normals are NumPy's bits; tail normals (0.03 %) go through log1p and may differ from a host's
 * NumPy in the last bit. */
int rocco_b200_numpy_normals_dev(unsigned long long seed_lo, unsigned long long seed_hi, unsigned long long skip,
                                 unsigned long long count, double *d_out, unsigned long long *words_consumed, void *cuda_stream);
/* Host: the PCG64 state default_rng(seed) starts from: out = {state low 64, state high 64, inc low 64, inc high 64}. */
int rocco_b200_numpy_seed_state(unsigned long long seed_lo, unsigned long long seed_hi, unsigned long long out[4]);
/* Words per chunk of the parallel parse (default 64, clamped to 1 .. 256; <= 0: the default); results do not change.
 * Returns the previous value. */
int rocco_b200_numpy_streams_set_chunk_words(int words);
/* _estimate_effective_sample_size (inference.py:446-501) of a host series. */
int rocco_effective_sample_size_f64(const double *values, size_t n, int max_lag, double *n_eff, double *tau_int,
                                    int *lags_used);
/* Median and count of the scores > 0 (rocco.py:762-769, the scale of the automatic gamma); NaNs sort last and would
 * count as positive, so the caller rejects non-finite scores first, as rocco.py:1019-1020 does. */
int rocco_positive_score_median_f64(const double *scores, size_t n, double *median, long long *count);

/* ------------------------------------------------------------------ column statistics */
enum {
    ROCCO_STAT_MEDIAN = 0,     /* np.median                                   (rocco.py:265)  */
    ROCCO_STAT_QUANTILE = 1,   /* np.quantile(method="nearest"), arg0 = q     (rocco.py:267)  */
    ROCCO_STAT_TMEAN = 2,      /* nearest-rank trimmed mean, arg0 = tprop     (rocco.py:273)  */
    ROCCO_STAT_MEAN = 3,       /*                                             (rocco.py:299)  */
    ROCCO_STAT_MAD = 4,        /* median |x - median|, scale 1                (rocco.py:325)  */
    ROCCO_STAT_IQR = 5,        /* percentile(arg1) - percentile(arg0), linear (rocco.py:327)  */
    ROCCO_STAT_STD = 6,        /* ddof 0                                      (rocco.py:329)  */
    ROCCO_STAT_TSTD = 7        /* ddof 1 inside nearest-rank limits, arg0 = tprop (rocco.py:331) */
};
int rocco_column_stat_f64(const double *matrix, size_t m, size_t n, int stat,
                          double arg0, double arg1, double power, double *out);
int rocco_b200_column_stat_dev(const void *d_matrix, int dtype, size_t m, size_t n, int stat,
                               double arg0, double arg1, double power, double *d_out, void *cuda_stream);
/* Column-statistics kernel choice: 1 = the shared-memory tile kernel (radix select per rank) for every m >= 2, any other
 * value = automatic (per-thread lists below the measured crossover, the tile kernel from it on and wherever the lists
 * do not fit).  Both give the same values; returns the previous mode. */
int rocco_b200_colstat_set_mode(int mode);

/* ------------------------------------------------------------------ matrix assembly / input staging (SURVEY.md 8(f) rank 3)
 * The step BEFORE the hot path, on the device, so that what crosses PCIe is the decoded alignment records (or the
 * float32 per-bin coverage), not the float64 samples x bins matrix.  BAM/BGZF decoding itself stays with htslib. */
typedef struct rocco_b200_count_options {        /* the fields of ccounts_countOptions the coverage loop reads (ccounts_backend.h:59-75) */
    int32_t flag_include, flag_exclude, min_mapping_quality, paired_end_mode, one_read_per_bin, reserved;
    int64_t read_length, min_template_length, max_insert_size, shift_forward_strand53, shift_reverse_strand53, extend_bp;
} rocco_b200_count_options;
/* ccounts_backend.c:2416-2574: per-read filters, fragment inference, strand shifts / extension, clipping, one-read-per-bin,
 * delta buffer + prefix sum.  Records are device arrays (struct of arrays of what htslib decodes: bam1_core_t pos,
 * bam_endpos, flag, qual, isize, mtid == tid); d_counts [count_len] float32, count_len = ceil((end - start) / step). */
int rocco_b200_count_alignment_region_dev(const int64_t *d_pos, const int64_t *d_endpos, const uint16_t *d_flag,
                                          const uint8_t *d_mapq, const int64_t *d_isize, const uint8_t *d_mate_same_tid,
                                          size_t n_reads, const rocco_b200_count_options *options, int64_t start, int64_t end,
                                          int64_t step, float *d_counts, size_t count_len, void *cuda_stream);
typedef struct rocco_b200_track {                /* one sample's counted window */
    const float *d_counts;                       /* device, count_len bins from count_start                        */
    size_t count_len;
    int64_t count_start;                         /* multiple of step (readtracks.py:468)                           */
    double norm_scale;                           /* metadata["norm_scale"] (readtracks.py:495)                     */
    double const_scale;                          /* applied when >= 0 (readtracks.py:500-503)                      */
    int32_t scale_by_step;                       /* divide by step (readtracks.py:496-498)                         */
    int32_t reserved;
} rocco_b200_track;
/* readtracks.py:505-516: per track the first and last bin whose SCALED value is > 0 (host outputs; -1, -1: no data). */
int rocco_b200_track_positive_range_dev(const rocco_b200_track *tracks, int n_tracks, int64_t step, int64_t *first_bin_out,
                                        int64_t *last_bin_out, void *cuda_stream);
/* readtracks.py:492-518 + 590-633: rows = the tracks that have data (in order), columns = the sorted union of their
 * interval starts, given as `n_segments` maximal runs of consecutive bins (segment_start_bp, segment_first_column);
 * value = np.round(counts * norm_scale [/ step] [* const_scale], round_digits) inside the track's positive range, else 0.
 * d_matrix: [n_kept][n_columns] float64 (out_f32 = 0) or float32; d_intervals: [n_columns] int64 interval starts. */
int rocco_b200_assemble_matrix_dev(const rocco_b200_track *tracks, const int64_t *first_bin, const int64_t *last_bin,
                                   int n_tracks, int64_t step, int round_digits, const int64_t *segment_start_bp,
                                   const int64_t *segment_first_column, int n_segments, size_t n_columns, int out_f32,
                                   void *d_matrix, int64_t *d_intervals, void *cuda_stream);

#ifdef __cplusplus
}
#endif
#endif /* ROCCO_B200_H */
