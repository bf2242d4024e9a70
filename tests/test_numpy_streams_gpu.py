"""NumPy streams on the device (random_streams="numpy"): the generator against numpy.random.default_rng, the budget null
against the reference's goldens and its host-replayed streams, sample sharding and the default flow.

Exactness contract of the generator: the words consumed for N normals are NumPy's (a second generator advanced by
random_raw(words) reaches the same state), fast-path and wedge normals are bit-identical, and tail normals (|x| beyond
the ziggurat's R) are within 1 ulp -- they go through log1p, which NumPy takes from the host's libm.
"""
import ctypes
import json
import math
import os

import numpy as np
import pytest

from rocco_b200.synth import chrom_matrix_numpy
from tests.test_budget_gpu import COUNT_KEYS, CONTINUOUS_TOL, INDICATOR_KEYS, reference_innovations
from tests.test_budget_sharded_gpu import assert_close_details, run_shards

pytestmark = pytest.mark.gpu

M64 = (1 << 64) - 1
NOR_R = 3.6541528853610087963519472518
BIG_SEEDS = [0, 7 + 104729 * 3, 2**64 + 104729]
BIG_COUNT = 20_000_000
CHUNKS = [64, 32, 1, 2, 3, 5]
DISCRETE_KEYS = {"num_null_draws", "max_null_draws", "wild_bandwidth", "ess_lags_used", "ess_max_lag", "num_loci",
                 "negative_support_size", "positive_score_count"}
_REF = {}


def device_normals(seed, skip, count):
    import torch
    from rocco_b200 import _lib
    out = torch.empty(count, dtype=torch.float64, device="cuda")
    words = ctypes.c_ulonglong(0)
    st = _lib.load().rocco_b200_numpy_normals_dev(seed & M64, seed >> 64, skip, count, ctypes.c_void_p(out.data_ptr()),
                                                  ctypes.byref(words), ctypes.c_void_p(torch.cuda.current_stream().cuda_stream))
    _lib.check(st, "numpy normals")
    torch.cuda.synchronize()
    return out.cpu().numpy(), int(words.value)


def reference(seed, skip, count):
    key = (seed, skip, count)
    if key not in _REF:
        g = np.random.default_rng(seed)
        if skip:
            g.standard_normal(skip)
        want = g.standard_normal(count)
        _REF[key] = (want, g.bit_generator.state)
    return _REF[key]


def check_stream(seed, skip, count, got, words):
    """Contract 1-3; returns (tail normals that differ, tail normals)."""
    want, state = reference(seed, skip, count)
    g = np.random.default_rng(seed)
    g.bit_generator.random_raw(words)
    assert g.bit_generator.state == state, (seed, skip, count, words)
    diff = got.view(np.uint64) != want.view(np.uint64)
    tail = np.abs(want) > NOR_R
    assert not np.any(diff & ~tail), (seed, skip, count, np.flatnonzero(diff & ~tail)[:5])
    if np.any(diff):
        assert np.all(np.abs(got[diff] - want[diff]) <= np.spacing(np.abs(want[diff]))), (seed, skip, count)
    return int(np.sum(diff)), int(np.sum(tail))


@pytest.fixture
def chunk_words():
    from rocco_b200 import _lib
    lib = _lib.load()
    prev = lib.rocco_b200_numpy_streams_set_chunk_words(64)

    def set_(w):
        lib.rocco_b200_numpy_streams_set_chunk_words(int(w))
    yield set_
    lib.rocco_b200_numpy_streams_set_chunk_words(prev)


@pytest.mark.parametrize("chunk", CHUNKS)
@pytest.mark.parametrize("seed", BIG_SEEDS)
def test_normals_match_numpy(seed, chunk, chunk_words):
    chunk_words(chunk)
    got, words = device_normals(seed, 0, BIG_COUNT)
    differ, tails = check_stream(seed, 0, BIG_COUNT, got, words)
    print(f"seed={seed} chunk={chunk}: {tails} tail normals, {differ} differ from this host's NumPy in the last bit")
    # a window deep inside the stream: skip through two thirds of it
    skip = 2 * BIG_COUNT // 3 + 1
    got2, words2 = device_normals(seed, skip, 1001)
    want, _ = reference(seed, 0, BIG_COUNT)
    assert np.array_equal(got2.view(np.uint64), got[skip:skip + 1001].view(np.uint64))
    g = np.random.default_rng(seed)
    g.standard_normal(skip + 1001)
    h = np.random.default_rng(seed)
    h.bit_generator.random_raw(words2)
    assert h.bit_generator.state == g.bit_generator.state


@pytest.mark.parametrize("chunk", CHUNKS)
def test_skip_and_count_across_chunk_boundaries(chunk, chunk_words):
    chunk_words(chunk)
    block = 128 * chunk
    skips = sorted({0, 1, 3, chunk - 1 if chunk > 1 else 5, chunk + 1, block - 1, block + 1, 5 * block + 3, 33 * block + 7})
    counts = sorted({1, 2, max(1, chunk - 1), chunk, chunk + 1, block - 1, block + 1})
    for seed in (1, 2**32 + 11):
        for skip in skips:
            for count in counts:
                got, words = device_normals(seed, skip, count)
                check_stream(seed, skip, count, got, words)


def test_seed_sums_beyond_64_bits():
    got, words = device_normals(2**64 - 1 + 104729 * 4, 0, 5000)
    check_stream(2**64 - 1 + 104729 * 4, 0, 5000, got, words)


# ------------------------------------------------------------------ the estimator
@pytest.fixture(scope="module")
def budget_golden():
    return np.load(os.path.join(os.path.dirname(__file__), "golden", "reference_budget_v1_11_0.npz"))


@pytest.mark.parametrize("tag", ["ref_test", "synth_a", "synth_b"])
def test_numpy_streams_estimator_meets_the_reference(budget_golden, tag):
    from rocco_b200 import inference as inf
    g = budget_golden
    kw = json.loads(str(g[f"{tag}_kwargs"]))
    want = json.loads(str(g[f"{tag}_meta"]))
    centered, scores = g[f"{tag}_centered"], g[f"{tag}_scores"]
    m, n = centered.shape
    frac, meta = inf.estimate_budget_nonnull_fraction_from_wild_bootstrap_null(
        centered, observed_scores=scores, return_details=True, random_streams="numpy", **kw)
    # the gates of the replay test (test_budget_gpu.py), without handing the streams over
    assert set(want) <= set(meta)
    for k, v in want.items():
        if isinstance(v, (str, bool)):
            assert meta[k] == v, k
        elif k in INDICATOR_KEYS:
            assert abs(meta[k] - v) <= 2.0 / n + 1e-12, (k, meta[k], v)
        elif k in COUNT_KEYS:
            assert abs(meta[k] - v) <= 2.0 + 1e-6 * abs(v), (k, meta[k], v)
        else:
            assert abs(meta[k] - v) <= CONTINUOUS_TOL * max(1.0, abs(v)), (k, meta[k], v)
    assert abs(frac - float(g[f"{tag}_fraction"])) <= 2.0 / n
    # and the same call fed NumPy's own array
    bw = inf._resolve_budget_bootstrap_bandwidth(n, kw.get("dependence_lag_hint"))
    inn = reference_innovations(kw.get("random_seed", 0), kw["num_null_draws"], m, n, 2 * bw + 1)
    frac_i, meta_i = inf.estimate_budget_nonnull_fraction_from_wild_bootstrap_null(
        centered, observed_scores=scores, return_details=True, innovations=inn, **kw)
    assert set(meta) == set(meta_i)
    for k, v in meta_i.items():
        if isinstance(v, (str, bool, int)) or k in DISCRETE_KEYS:
            assert meta[k] == v, k
        else:
            assert abs(meta[k] - v) <= 1e-12 * max(abs(v), 1e-300) or meta[k] == v, (k, meta[k], v)
    assert frac == frac_i


def test_row_groups_continue_the_stream():
    """More than 256 MB of normals per draw: the rows are generated in groups, each continuing the stream."""
    import torch
    from rocco_b200 import pipeline
    from rocco_b200.inference import _resolve_budget_bootstrap_bandwidth
    m, n = 5, 7_000_000
    c = torch.from_numpy(np.random.default_rng(3).standard_normal((m, n))).cuda()
    bw = _resolve_budget_bootstrap_bandwidth(n, None)
    assert m * (n + 2 * bw) > (32 << 20)
    kw = dict(params=pipeline.score_params(prior_df=6.0), num_null_draws=2, min_null_draws=2, random_seed=9)
    got = pipeline._budget_null_sharded(c, m, 0, None, random_streams="numpy", **kw)
    inn = torch.from_numpy(reference_innovations(9, 2, m, n, 2 * bw + 1)).cuda()
    want = pipeline._budget_null_sharded(c, m, 0, None, innovations=inn, **kw)
    assert got[1]["num_null_draws"] == 2.0
    assert_close_details(got[1], want[1], n, rel=1e-12, what="row groups")


# ------------------------------------------------------------------ sample sharding
@pytest.fixture(scope="module")
def case():
    import torch
    from rocco_b200 import pipeline
    x = chrom_matrix_numpy(7, 60_000, seed=17)
    prm = pipeline.score_params(prior_df=6.0)
    scores, det = pipeline.score_loci_wls_device(torch.from_numpy(x).cuda(), params=prm, details=True)
    return {"centered": det["centered_matrix"], "scores": scores, "params": prm, "hint": det["local_baseline_window"]}


def test_three_plus_four_shards_match_the_unsharded_numpy_streams(case):
    from rocco_b200 import pipeline
    c, s, prm = case["centered"], case["scores"], case["params"]
    n = c.shape[1]
    common = dict(params=prm, dependence_lag_hint=case["hint"], num_null_draws=10, min_null_draws=10, random_seed=21,
                  random_streams="numpy")
    want_frac, want = pipeline.budget_null_device(c, s, **common)
    out = run_shards([(c[:3].contiguous(), 0, None), (c[3:].contiguous(), 3, None)], d_observed_scores=s, **common)
    assert [o[0] for o in out] == ["ok", "ok"], out
    (f0, d0), (f1, d1) = out[0][1], out[1][1]
    assert d0 == d1 and f0 == f1
    assert abs(f0 - want_frac) <= 2.0 / n
    assert_close_details(d0, want, n, what="3+4 shards, numpy streams")


def test_shard_rows_are_the_rows_of_the_whole_field(chunk_words):
    L, m = 60_000 + 2 * 39, 7
    seed = 21 + 104729 * 2
    whole, _ = device_normals(seed, 0, m * L)
    for chunk in (64, 3):
        chunk_words(chunk)
        for off, rows in ((0, 3), (3, 4), (5, 2)):
            part, _ = device_normals(seed, off * L, rows * L)
            assert np.array_equal(part.view(np.uint64), whole[off * L:(off + rows) * L].view(np.uint64)), (chunk, off)


# ------------------------------------------------------------------ the default flow
SMALL_GENOME = ["chrX1", "chrX2", "chrX3"]
SMALL_SIZES = [20_000, 31_013, 40_000]
SMALL_SAMPLES = 6


@pytest.fixture(scope="module")
def small():
    import torch
    xs = [chrom_matrix_numpy(SMALL_SAMPLES, n, seed=301 + k) for k, n in enumerate(SMALL_SIZES)]
    return xs, [torch.from_numpy(x).cuda() for x in xs]


def _hand_nulls(mats, prm, streams):
    from rocco_b200 import pipeline
    from rocco_b200.inference import _resolve_local_baseline_window
    nulls, scores, cents, windows = {}, {}, {}, {}
    for c, x in zip(SMALL_GENOME, mats):
        s, extra = pipeline.score_loci_wls_device(x, params=prm, details=True)
        w = _resolve_local_baseline_window(x.shape[1], 101)
        _, nulls[c] = pipeline.budget_null_device(extra["centered_matrix"], s, params=prm, dependence_lag_hint=w,
                                                  num_null_draws=25, random_seed=0, random_streams=streams)
        scores[c], cents[c], windows[c] = s, extra["centered_matrix"], w
    return nulls, scores, cents, windows


def test_default_flows_equal_the_hand_composition(small):
    import torch
    from rocco_b200 import pipeline
    from rocco_b200.rocco import _resolve_budgets, _resolve_chrom_gamma
    _, mats = small
    prm = pipeline.score_params(prior_df=6.0)
    args = {"random_streams": "numpy"}
    nulls, scores, _, _ = _hand_nulls(mats, prm, "numpy")
    budgets, meta = _resolve_budgets({c: {"budget_count_hat": nulls[c]["effective_count"],
                                          "total_count": nulls[c]["effective_total_count"]} for c in SMALL_GENOME},
                                     pipeline._default_flow_args(args))
    gammas = {c: _resolve_chrom_gamma(c, {"gamma": None}, None, nulls[c])[0] for c in SMALL_GENOME}
    want = pipeline.run_shard(mats, [budgets[c] for c in SMALL_GENOME], [gammas[c] for c in SMALL_GENOME], params=prm)
    got = pipeline.run_shard(mats, None, None, params=prm, chrom_names=SMALL_GENOME, genome_names=SMALL_GENOME,
                             default_args=args)
    assert got["defaults"]["null"] == [nulls[c] for c in SMALL_GENOME]
    assert got["budgets"] == [budgets[c] for c in SMALL_GENOME] and got["gammas"] == [gammas[c] for c in SMALL_GENOME]
    assert torch.equal(got["d_masks"], want["d_masks"]) and got["results"] == want["results"]
    # the Philox default flow differs: the streams are really switched
    philox = pipeline.run_shard(mats, None, None, params=prm, chrom_names=SMALL_GENOME, genome_names=SMALL_GENOME)
    assert philox["defaults"]["null"] != got["defaults"]["null"]
    # samples over ranks, one process
    ss = pipeline.run_sample_sharded_defaults(iter(zip(SMALL_GENOME, mats)), SMALL_SAMPLES, prm, default_args=args)
    snulls = {}
    for c, x in zip(SMALL_GENOME, mats):
        s, cent, window = pipeline.score_loci_wls_sample_sharded(x, SMALL_SAMPLES, prm, keep_centered=True)
        _, snulls[c] = pipeline.budget_null_sample_sharded(cent, s, params=prm, dependence_lag_hint=window,
                                                           random_streams="numpy")
    sb, smeta = _resolve_budgets({c: {"budget_count_hat": snulls[c]["effective_count"],
                                      "total_count": snulls[c]["effective_total_count"]} for c in SMALL_GENOME},
                                 pipeline._default_flow_args(args))
    assert ss["defaults"]["null"] == snulls and ss["budgets"] == sb and ss["defaults"]["budget_meta"] == smeta
    assert ss["gammas"] == {c: _resolve_chrom_gamma(c, {"gamma": None}, None, snulls[c])[0] for c in SMALL_GENOME}


def test_default_flow_budgets_and_gammas_match_the_oracle(small):
    from oracle import budget as ob
    from rocco_b200 import pipeline
    from rocco_b200.rocco import _resolve_budgets, _resolve_chrom_gamma
    _, mats = small
    prm = pipeline.score_params(prior_df=6.0)
    args = pipeline._default_flow_args({"random_streams": "numpy"})
    got = pipeline.run_shard(mats, None, None, params=prm, chrom_names=SMALL_GENOME, genome_names=SMALL_GENOME,
                             default_args={"random_streams": "numpy"})
    _, scores, cents, windows = _hand_nulls(mats, prm, "numpy")
    onulls, oscores = {}, {}
    for c in SMALL_GENOME:
        oscores[c] = scores[c].cpu().numpy()
        _, onulls[c] = ob.estimate_budget_nonnull_fraction(cents[c].cpu().numpy(), observed_scores=oscores[c],
                                                           dependence_lag_hint=windows[c], return_details=True, prior_df=6.0,
                                                           num_null_draws=25, random_seed=0)
    ob_budgets, _ = _resolve_budgets({c: {"budget_count_hat": onulls[c]["effective_count"],
                                          "total_count": onulls[c]["effective_total_count"]} for c in SMALL_GENOME}, args)
    for k, c in enumerate(SMALL_GENOME):
        og = _resolve_chrom_gamma(c, {"gamma": None}, oscores[c], onulls[c])[0]
        assert onulls[c]["num_null_draws"] == got["defaults"]["null"][k]["num_null_draws"], c
        assert abs(got["budgets"][k] - ob_budgets[c]) <= 1e-6 * ob_budgets[c], (c, got["budgets"][k], ob_budgets[c])
        assert abs(got["gammas"][k] - og) <= 1e-6 * og, (c, got["gammas"][k], og)
        n = SMALL_SIZES[k]
        assert pipeline.target_count_for_budget(n, got["budgets"][k]) == math.floor(n * ob_budgets[c]), c


# ------------------------------------------------------------------ defaults and rejections
def test_explicit_philox_is_the_default(case):
    from rocco_b200 import pipeline
    c, s, prm = case["centered"], case["scores"], case["params"]
    kw = dict(params=prm, dependence_lag_hint=case["hint"], num_null_draws=6, random_seed=4)
    assert pipeline.budget_null_device(c, s, random_streams="philox", **kw) == pipeline.budget_null_device(c, s, **kw)
    assert pipeline.budget_null_sample_sharded(c, s, random_streams="philox", **kw) == pipeline.budget_null_sample_sharded(c, s, **kw)


def test_random_streams_rejections(case):
    import torch
    from rocco_b200 import inference, pipeline
    c, s, prm = case["centered"], case["scores"], case["params"]
    m, n = c.shape
    with pytest.raises(ValueError):
        pipeline.budget_null_device(c, s, params=prm, random_streams="pcg64")
    with pytest.raises(ValueError):
        pipeline.budget_null_device(c, s, params=prm, random_streams="numpy", random_seed=-1)
    with pytest.raises(ValueError):
        pipeline.budget_null_sample_sharded(c, s, params=prm, random_streams="numpy", random_seed=-2)
    inn = torch.zeros((1, m, n + 2 * 39), dtype=torch.float64, device="cuda")
    with pytest.raises(ValueError):
        pipeline._budget_null_sharded(c, m, 0, None, params=prm, num_null_draws=1, innovations=inn, random_streams="numpy")
    x = c[:2, :500].cpu().numpy()
    with pytest.raises(ValueError):
        inference.estimate_budget_nonnull_fraction_from_wild_bootstrap_null(x, random_streams="numpy",
                                                                            innovations=np.zeros((25, 2, 520)))
    with pytest.raises(ValueError):
        inference.estimate_budget_nonnull_fraction_from_wild_bootstrap_null(x, random_streams="bogus")
    with pytest.raises(ValueError):
        pipeline.run_shard([torch.from_numpy(chrom_matrix_numpy(4, 5000, seed=1)).cuda()], None, None, params=prm,
                           chrom_names=["chrQ"], default_args={"random_streams": "mt"})
