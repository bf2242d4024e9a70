"""GPU parity: scoring chain (log2p1 -> pilot -> cross-fit Whittaker baseline -> centered WLS) vs the oracle.

Floating-point gate (BASELINE.json north_star / SURVEY.md 8d): max relative error <= 1e-5 with
denominator max(|ref|, 1e-3).  Observed errors are orders of magnitude smaller; the tighter asserts
below (1e-6) guard against regressions while staying above the reference's own ~1e-10 solver noise.
"""
import numpy as np
import pytest

from rocco_b200.synth import chrom_matrix_numpy
from tests.conftest import rel_err

pytestmark = pytest.mark.gpu

TOL = 1e-5          # the stated tolerance
TIGHT = 1e-6        # regression guard (abs error ~1e-10 = the Whittaker solve noise floor, over the 1e-3 denominator floor)

DETAIL_KEYS = ("mean", "raw_variance", "prior_variance", "moderated_variance", "standard_error", "z_scores")


@pytest.fixture(scope="module")
def rb():
    import rocco_b200
    return rocco_b200


def _check_details(got, want, tol=TIGHT):
    for k in DETAIL_KEYS:
        e = rel_err(got[k], want[k])
        assert e <= tol, (k, e)


# ------------------------------------------------------------------ golden vectors from the real reference
@pytest.mark.parametrize("tag,kw", [("a", {}),
                                    ("b", dict(prior_df=6.0, lower_bound_z=0.5, precision_floor_ratio=0.05)),
                                    ("c", dict(min_effect=0.25))])
def test_score_loci_wls_matches_reference_golden(rb, golden, tag, kw):
    sc, det = rb.score_loci_wls(golden["score_x"], return_details=True, **kw)
    assert sc.dtype == np.float64 and sc.shape == (3000,)
    assert rel_err(sc, golden[f"score_{tag}_scores"]) <= TIGHT
    for k in DETAIL_KEYS:
        assert rel_err(det[k], golden[f"score_{tag}_{k}"]) <= TIGHT, k
    if tag == "a":
        meta = golden["score_a_meta"]
        assert det["input_scale"] == "log2p1"
        assert det["local_baseline_window"] == 101 and det["local_baseline_lambda"] == meta[1]
        assert det["prior_spatial_window"] == 31 and det["degrees_of_freedom"][0] == meta[3]
        assert np.max(np.abs(det["centered_matrix"] - golden["score_a_centered"])) <= 1e-8


def test_float32_input_matches_reference_golden(rb, golden):
    sc = rb.score_loci_wls(golden["score_x"].astype(np.float32))
    assert rel_err(sc, golden["score_f32_scores"]) <= TIGHT


@pytest.mark.parametrize("tag", ["n2", "n3", "n4", "n24", "n25", "n130"])
def test_small_n_branches_match_reference_golden(rb, golden, tag):
    sc, det = rb.score_loci_wls(golden[f"small_{tag}_x"], lower_bound_z=0.0, return_details=True)
    assert rel_err(sc, golden[f"small_{tag}_scores"]) <= TIGHT
    assert rel_err(det["mean"], golden[f"small_{tag}_mean"]) <= TIGHT
    assert rel_err(det["standard_error"], golden[f"small_{tag}_se"]) <= TIGHT


# ------------------------------------------------------------------ the reference's own known answers
def test_known_answer_log_scale(rb):
    """reference tests/test_rocco.py:234-246"""
    scores, details = rb.score_loci_wls(np.array([[1.0, 15.0]]), lower_bound_z=0.0, return_details=True)
    assert details["input_scale"] == "log2p1"
    assert "sample_intercepts" not in details and "sample_baselines" not in details
    assert np.allclose(details["mean"], np.array([-1.5, 1.5]))
    assert np.allclose(details["z_scores"], np.array([-0.67449076, 0.67449076]))
    assert np.allclose(scores, np.array([-0.67449076, 0.67449076]))


def test_known_answer_min_effect(rb):
    """reference tests/test_rocco.py:249-258"""
    scores, details = rb.score_loci_wls(np.array([[1.0, 15.0]]), min_effect=0.5, return_details=True)
    assert np.isclose(details["min_effect"], 0.5)
    assert scores[1] < details["z_scores"][1] and scores[0] < details["z_scores"][0]


def test_known_answer_precision_floor(rb):
    """reference tests/test_rocco.py:261-285"""
    from rocco_b200 import inference
    centered = np.array([[0.05, 1.0, 1.0, 0.05], [0.04, 1.0, 1.0, 0.04], [0.06, 1.0, 1.0, 0.06]], dtype=np.float64)
    lo_s, lo_d = inference._score_centered_wls_matrix(centered, prior_df=6.0, precision_floor_ratio=0.0)
    hi_s, hi_d = inference._score_centered_wls_matrix(centered, prior_df=6.0, precision_floor_ratio=0.25)
    assert np.isclose(hi_d["precision_floor_ratio"], 0.25)
    assert np.all(hi_d["standard_error"] >= lo_d["standard_error"]) and np.all(hi_s <= lo_s)


def test_known_answer_low_memory_dtype(rb):
    """reference tests/test_rocco.py:288-297"""
    scores, details = rb.score_loci_wls(np.array([[1.0, 3.0, 7.0], [1.2, 2.8, 6.5]]), low_memory=True, return_details=True)
    assert scores.dtype == np.float64 and details["centered_matrix"].dtype == np.float32
    assert np.all(np.isfinite(details["centered_matrix"]))


def test_known_answer_tied_large_matrix(rb):
    """reference tests/test_rocco.py:331-345: 3 x 250000 zeros (all-ties path through the order statistics)"""
    from rocco_b200 import inference
    scores, details = inference._score_centered_wls_matrix(np.zeros((3, 250000)), lower_bound_z=1.0, prior_df=5.0)
    assert scores.shape == (250000,)
    assert np.allclose(details["mean"], 0.0) and np.allclose(details["z_scores"], 0.0) and np.allclose(scores, -1.0)
    assert np.all(details["standard_error"] > 0.0)


def test_known_answer_noisy_track_downweighted(rb):
    """reference tests/test_rocco.py:348-375"""
    from rocco_b200 import inference
    x = np.linspace(-4.0, 4.0, 513, dtype=np.float64)
    smooth = 0.9 * np.sin(x) + 0.15 * np.cos(2.0 * x)
    noisy = smooth.copy()
    region = slice(180, 333)
    noisy[region] += 0.75 * np.where((np.arange(region.stop - region.start) % 2) == 0, 1.0, -1.0)
    centered = np.vstack([smooth, noisy])
    _, details = inference._score_centered_wls_matrix(centered, lower_bound_z=0.0, prior_df=6.0, spatial_window=31)
    simple_mean = centered.mean(axis=0)
    quiet = slice(40, 140)
    assert np.mean(np.abs(details["mean"][region] - smooth[region])) < np.mean(np.abs(simple_mean[region] - smooth[region]))
    assert np.mean(details["standard_error"][region]) > np.mean(details["standard_error"][quiet])


def test_known_answer_crossfit_baseline_tracks_broad_background(rb, golden):
    """reference tests/test_rocco.py:378-394"""
    from rocco_b200 import inference
    y = golden["base129_y"]
    baseline = inference._consenrich_crossfit_whittaker_baseline(y, block_size=41)
    assert baseline.shape == y.shape
    assert np.max(np.abs(baseline - golden["base129_out"])) <= 1e-9
    x = np.arange(129, dtype=np.float64)
    broad = 2.5 * np.exp(-0.5 * ((x - 64.0) / 18.0) ** 2)
    residual = y - baseline
    assert baseline[46] > 0.5 * broad[46]
    assert residual[64] > 3.0 * max(residual[46], 1.0e-6)


# ------------------------------------------------------------------ stage-level parity
def test_stage_baseline_matches_reference_golden(rb, golden):
    from rocco_b200 import inference
    base, window, lam = inference._estimate_local_background_matrix(golden["base_y"])
    assert window == 101 and lam == inference._consenrich_whittaker_lambda(101) == golden["score_a_meta"][1]
    assert np.max(np.abs(base - golden["base_out"])) <= 1e-8


@pytest.mark.parametrize("n", [25, 26, 101, 1279, 2561, 4104, 4105, 9728, 9729, 12288, 25000, 140001])
def test_baseline_matches_oracle_across_tile_and_table_edges(rb, oracle, n):
    """sizes straddle the head table (4096 + 8), the tile (9728) and the region (12288) boundaries"""
    from rocco_b200 import _baseline
    rng = np.random.default_rng(n)
    y = rng.normal(size=(2, n)) + 2.0 * np.sin(np.arange(n) / 700.0) + (rng.random((2, n)) < 0.01) * 6.0
    lam = oracle.whittaker_lambda(oracle.resolve_local_baseline_window(n))
    want = oracle.native("port").crossfit_whittaker_baseline(y, lam)
    got = _baseline.crossfit_whittaker_baseline(y, lam)
    assert got.shape == want.shape
    assert np.max(np.abs(got - want)) <= 2e-9, float(np.max(np.abs(got - want)))
    got1 = _baseline.crossfit_whittaker_baseline(y[0], lam)
    assert got1.shape == (n,) and np.max(np.abs(got1 - want[0])) <= 2e-9


# (3, 20741) has no steady tile and (3, 20742) exactly one; one row gives a single alignment group; 24 rows of 300007 or
# 300008 bins and 4 rows of 1000003 give each persistent cluster several tiles, so both landing buffers and both phases
# of every mbarrier are used (odd n: two row groups with different bulk-copy shifts, even n: one)
@pytest.mark.parametrize("rows,n", [(3, 140001), (5, 60002), (2, 300007), (1, 140001), (3, 20741), (3, 20742),
                                    (24, 300007), (24, 300008), (4, 1000003)])
def test_streaming_steady_tile_kernel_matches_the_oracle(rb, oracle, rows, n):
    """the streaming cluster-pair kernel of the interior tiles within 2e-9 of the oracle, odd row lengths (every 16-byte
    alignment class of the bulk copies), the row lengths at which the first steady tile appears, and launches in which
    each cluster walks several tiles"""
    from rocco_b200 import _baseline
    rng = np.random.default_rng(300 + rows)
    y = rng.normal(size=(rows, n)) + 2.0 * np.sin(np.arange(n) / 900.0) + (rng.random((rows, n)) < 0.01) * 6.0
    lam = oracle.whittaker_lambda(oracle.resolve_local_baseline_window(n))
    want = oracle.native("port").crossfit_whittaker_baseline(y, lam)
    got = _baseline.crossfit_whittaker_baseline(y, lam)
    assert np.max(np.abs(got - want)) <= 2e-9, float(np.max(np.abs(got - want)))


@pytest.mark.parametrize("n", [250000, 250001, 250002, 250003])
def test_float32_rows_of_every_alignment_class_match_float64_storage(rb, n):
    """float32 storage: four row-alignment classes for the 16-byte bulk copies (row length mod 4).  The reference widens to
    float64 first (inference.py:40-47), so the same values stored either way must score alike: bit for bit when the rows of
    both layouts fall in the same alignment class (n a multiple of 4: identical tile regions), and within the halo
    truncation (1e-11) otherwise, where the regions start a few bins apart."""
    import torch
    from rocco_b200 import pipeline
    from rocco_b200.synth import chrom_matrix_torch
    dev = torch.device("cuda", 0)
    x32 = chrom_matrix_torch(5, n, 7 + n % 5, dev, torch.float32)
    prm = pipeline.score_params(prior_df=6.0)
    s32, d32 = pipeline.score_loci_wls_device(x32, params=prm, details=True)
    s64, d64 = pipeline.score_loci_wls_device(x32.to(torch.float64), params=prm, details=True)
    if n % 4 == 0:
        assert torch.equal(d32["centered_matrix"], d64["centered_matrix"]) and torch.equal(s32, s64)
    else:
        assert float((d32["centered_matrix"] - d64["centered_matrix"]).abs().max()) <= 1e-11
        assert float((s32 - s64).abs().max()) <= 1e-9 * max(1.0, float(s64.abs().max()))


def test_baseline_small_n_is_zero(rb):
    from rocco_b200 import _baseline
    assert np.array_equal(_baseline.crossfit_whittaker_baseline(np.arange(24.0), 5.0), np.zeros(24))
    with pytest.raises(ValueError):
        _baseline.crossfit_whittaker_baseline(np.zeros((2, 2, 2)), 1.0)


def test_stage_centered_wls_matches_reference_golden(rb, golden):
    from rocco_b200 import inference
    sc, det = inference._score_centered_wls_matrix(golden["wls_centered"], prior_df=6.0, spatial_window=31)
    assert rel_err(sc, golden["wls_scores"]) <= TIGHT
    for k in ("mean", "raw_variance", "prior_variance", "moderated_variance", "standard_error"):
        assert rel_err(det[k], golden[f"wls_{k}"]) <= TIGHT, k


def test_wls_native_signature_and_errors(rb):
    from rocco_b200 import _wls
    out = _wls.score_centered_wls(np.random.default_rng(0).normal(size=(3, 64)), prior_df=6.0)
    assert len(out) == 8 and isinstance(out[6], float) and isinstance(out[7], int)
    assert out[6] == 28.0 + 6.0 and out[7] == 31
    with pytest.raises(ValueError):
        _wls.score_centered_wls(np.zeros(5))
    with pytest.raises(ValueError):
        rb.score_loci_wls(np.array([[1.0, np.nan, 2.0]]))
    with pytest.raises(ValueError):
        rb.score_loci_wls(np.zeros((0, 5)))
    with pytest.raises(ValueError):
        rb.score_loci_wls(np.zeros(5))


@pytest.mark.parametrize("window", [5, 7, 30, 31, 64, 201])
def test_spatial_windows_match_oracle(rb, oracle, window):
    from rocco_b200 import inference
    rng = np.random.default_rng(window)
    c = rng.normal(size=(3, 3000)) * (0.2 + np.abs(np.sin(np.arange(3000) / 150.0)))
    want_s, want = oracle.score_centered_wls_matrix(c, spatial_window=window)
    got_s, got = inference._score_centered_wls_matrix(c, spatial_window=window)
    assert got["prior_spatial_window"] == want["prior_spatial_window"]
    assert rel_err(got_s, want_s) <= TIGHT
    _check_details(got, want)


# ------------------------------------------------------------------ order statistics: multi-select == sort path
@pytest.mark.parametrize("m,n,seed,ties", [(3, 5, 1, True), (2, 37, 2, True), (4, 999, 3, True), (3, 20_000, 4, True),
                                           (3, 20_000, 6, False), (6, 300_000, 5, False)])
def test_trend_multiselect_equals_sort_path_bitwise(rb, m, n, seed, ties):
    """both paths compute exact order statistics, so every output must agree bit for bit"""
    from rocco_b200 import _lib, inference
    lib = _lib.load()
    rng = np.random.default_rng(seed)
    c = rng.normal(size=(m, n)) * (0.2 + np.abs(np.sin(np.arange(n) / 150.0)))
    if ties:
        c[:, : n // 3] = np.round(c[:, : n // 3], 2)          # ties in |signal|
    prev = lib.rocco_b200_trend_set_mode(1)
    try:
        want_s, want = inference._score_centered_wls_matrix(c, prior_df=6.0)
    finally:
        lib.rocco_b200_trend_set_mode(0)
    fb0 = lib.rocco_b200_trend_fallback_rows()
    got_s, got = inference._score_centered_wls_matrix(c, prior_df=6.0)
    lib.rocco_b200_trend_set_mode(prev)
    assert np.array_equal(got_s, want_s)
    for k in DETAIL_KEYS:
        assert np.array_equal(got[k], want[k]), k
    if not ties:
        assert lib.rocco_b200_trend_fallback_rows() == fb0       # the fast path really ran


def test_trend_large_rows_take_the_fine_bucket_geometry_and_stay_exact(rb):
    """Rows longer than 6 M bins (hg38 @ 20 bp: chr1 has 12.4 M) switch to 2048 |signal| buckets / 128 variance buckets per
    octave so that no bucket outgrows its slot; the result must still equal the sort path bit for bit, without fallback."""
    from rocco_b200 import _lib, inference
    lib = _lib.load()
    rng = np.random.default_rng(11)
    m, n = 2, 12_500_000
    c = rng.normal(size=(m, n)) * (0.25 + 0.1 * np.abs(np.sin(np.arange(n) / 5000.0)))
    c[1] *= rng.standard_normal(n)                     # a bootstrap-like row: much mass near zero
    prev = lib.rocco_b200_trend_set_mode(1)
    try:
        want_s, want = inference._score_centered_wls_matrix(c, prior_df=6.0)
    finally:
        lib.rocco_b200_trend_set_mode(0)
    fb0 = lib.rocco_b200_trend_fallback_rows()
    got_s, got = inference._score_centered_wls_matrix(c, prior_df=6.0)
    lib.rocco_b200_trend_set_mode(prev)
    assert lib.rocco_b200_trend_fallback_rows() == fb0
    assert np.array_equal(got_s, want_s)
    for k in DETAIL_KEYS:
        assert np.array_equal(got[k], want[k]), k


def test_trend_fallback_on_massive_ties(rb):
    from rocco_b200 import _lib, inference
    lib = _lib.load()
    fb0 = lib.rocco_b200_trend_fallback_rows()
    c = np.zeros((2, 50_000))
    c[1, ::7] = 0.5
    sc, det = inference._score_centered_wls_matrix(c)
    assert lib.rocco_b200_trend_fallback_rows() > fb0            # over-capacity buckets -> sort path
    assert np.all(np.isfinite(sc))


# ------------------------------------------------------------------ end-to-end at benchmark-like shapes
@pytest.mark.parametrize("m,n,seed", [(10, 60_000, 21), (4, 250_000, 19), (25, 30_011, 5)])
def test_score_loci_wls_matches_oracle(rb, oracle, m, n, seed):
    x = chrom_matrix_numpy(m, n, seed=seed)
    want_s, want = oracle.score_loci_wls(x, prior_df=6.0, return_details=True)
    got_s, got = rb.score_loci_wls(x, prior_df=6.0, return_details=True)
    e = rel_err(got_s, want_s)
    assert e <= TOL and e <= TIGHT, e
    _check_details(got, want)
    assert np.max(np.abs(got["centered_matrix"] - want["centered_matrix"])) <= 1e-8


def test_score_then_solve_gives_reference_mask(rb, oracle):
    """the whole path on a chr21-like slice: GPU scores -> GPU solve must select the same bins as the
    oracle's scores -> oracle's solve (budget 0.02, gamma 1.0: hg_params chr21)"""
    x = chrom_matrix_numpy(10, 120_000, seed=2100)
    want_scores = oracle.score_loci_wls(x, prior_df=6.0)
    got_scores = rb.score_loci_wls(x, prior_df=6.0)
    want_sol, want_obj, want = oracle.solve_chrom_exact(want_scores, budget=0.02, gamma=1.0, return_details=True)
    got_sol, got_obj, got = rb.solve_chrom_exact(got_scores, budget=0.02, gamma=1.0, return_details=True)
    assert np.array_equal(got_sol, want_sol), int(np.sum(got_sol != want_sol))
    assert got["selected_count"] == want["selected_count"]
    assert abs(got_obj - want_obj) <= 1e-6 * abs(want_obj)
    assert abs(got["selection_penalty"] - want["selection_penalty"]) <= 1e-6


def test_sample_sharded_scoring_matches_unsharded(rb, oracle):
    """SURVEY.md 8e(2): per-sample stages on each shard, sum of the [4, bins] accumulators (the all-reduce, emulated
    here by adding the two shards' tensors on one GPU), then the per-bin finalisation."""
    import torch
    from rocco_b200 import pipeline
    x = chrom_matrix_numpy(12, 50_000, seed=77)
    prm = pipeline.score_params(prior_df=6.0)
    d = torch.from_numpy(x).cuda()
    acc = pipeline.score_partial_device(d[:5].contiguous(), prm) + pipeline.score_partial_device(d[5:].contiguous(), prm)
    got = pipeline.score_finalize_device(acc, 12, prm, details=True)
    want_s, want = oracle.score_loci_wls(x, prior_df=6.0, return_details=True)
    assert rel_err(got["scores"].cpu().numpy(), want_s) <= TIGHT
    for k in ("mean", "raw_variance", "prior_variance", "moderated_variance", "standard_error"):
        assert rel_err(got[k].cpu().numpy(), want[k]) <= TIGHT, k
    whole = pipeline.score_loci_wls_device(d, params=prm).cpu().numpy()
    assert np.max(np.abs(got["scores"].cpu().numpy() - whole)) <= 1e-12 * max(1.0, float(np.max(np.abs(whole))))
    # world size 1: the sharded entry is the unsharded computation
    one = pipeline.score_loci_wls_sample_sharded(d, 12, prm).cpu().numpy()
    assert np.max(np.abs(one - whole)) <= 1e-12 * max(1.0, float(np.max(np.abs(whole))))
