"""The slot collection (T3) of the trend's multi-select reading the 32-bit pair keys the fused rolling-variance pass
leaves (trend mode 0) against the sort path (mode 1).  Both are exact order statistics, so every output must agree bit
for bit.  The rows cover both bucket geometries (variance bits shifted by 46 up to 6 M bins, by 45 above), partial last
chunks and tiles, slot buckets holding thousands of tied pairs, and an all-zero row that falls back to the sort path
next to rows that do not."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

DETAIL_KEYS = ("mean", "raw_variance", "prior_variance", "moderated_variance", "standard_error", "z_scores")


def _wavy(rng, m, n):
    return rng.normal(size=(m, n)) * (0.2 + np.abs(np.sin(np.arange(n) / 150.0)))


def _run_modes(c, window):
    """scores and details of modes 1 and 0, and the fallback rows mode 0 added"""
    from rocco_b200 import _lib, inference
    lib = _lib.load()
    out, fb = {}, {}
    prev = lib.rocco_b200_trend_set_mode(0)
    try:
        for mode in (1, 0):
            lib.rocco_b200_trend_set_mode(mode)
            fb0 = lib.rocco_b200_trend_fallback_rows()
            out[mode] = inference._score_centered_wls_matrix(c, prior_df=6.0, spatial_window=window)
            fb[mode] = lib.rocco_b200_trend_fallback_rows() - fb0
    finally:
        lib.rocco_b200_trend_set_mode(prev)
    return out, fb


def _assert_identical(out, window):
    want_s, want = out[1]
    got_s, got = out[0]
    assert got["prior_spatial_window"] == window
    assert np.array_equal(got_s, want_s)
    for k in DETAIL_KEYS:
        assert np.array_equal(got[k], want[k]), k


@pytest.mark.parametrize("window", [31, 65])
@pytest.mark.parametrize("n", [2 * 131072 + 12345, 6_200_017])     # up to 6 M bins: yshift 46; above: yshift 45
def test_key_collection_equals_sort_path(window, n):
    rng = np.random.default_rng(n + window)
    m = 3 if n < 1_000_000 else 2
    c = _wavy(rng, m, n)
    out, fb = _run_modes(c, window)
    assert fb[0] == 0                                                 # the multi-select really ran on every row
    _assert_identical(out, window)


@pytest.mark.parametrize("window", [31, 65])
def test_key_collection_with_thousands_of_tied_pairs_per_slot(window):
    """a third of every row sits on 40 values, about 3000 pairs each (either sign): bin boundaries and medians fall
    into buckets holding thousands of identical |signal| values, still under the 8192-pair slot capacity"""
    rng = np.random.default_rng(100 + window)
    m, n = 3, 400_001
    c = _wavy(rng, m, n)
    ties = rng.uniform(0.05, 2.0, size=40)
    for r in range(m):
        idx = rng.permutation(n)[: 40 * 3000]
        c[r, idx] = np.repeat(ties, 3000) * rng.choice([-1.0, 1.0], size=idx.size)
    out, fb = _run_modes(c, window)
    assert fb[0] == 0                                                 # no row left the multi-select
    _assert_identical(out, window)


def test_key_collection_next_to_a_fallback_row():
    """an all-zero row overflows its slot and takes the sort path; the rows sharing its launches do not"""
    rng = np.random.default_rng(5)
    m, n = 3, 2 * 131072 + 777
    c = _wavy(rng, m, n)
    c[1] = 0.0
    out, fb = _run_modes(c, 31)
    assert fb[0] == 1
    _assert_identical(out, 31)


def test_trend_mode_mapping_keeps_only_the_sort_mode():
    from rocco_b200 import _lib
    lib = _lib.load()
    prev = lib.rocco_b200_trend_set_mode(1)
    try:
        assert lib.rocco_b200_trend_set_mode(1) == 1                  # 1 is kept
        for other in (0, 2, 7, -1):                                   # 0, and any other value, means 0
            lib.rocco_b200_trend_set_mode(other)
            assert lib.rocco_b200_trend_set_mode(1) == 0, other
    finally:
        lib.rocco_b200_trend_set_mode(prev)
