"""The fused rolling-variance kernel against the sort path's separate variance kernel, on rows long enough for
whole interior tiles, several chunks per row and a partial last chunk and tile.  Both kernels sum each block of 8
outputs the same way, so the scores and every detail vector must agree bit for bit, for the compiled default window
and for runtime windows up to the fused kernel's largest."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

DETAIL_KEYS = ("mean", "raw_variance", "prior_variance", "moderated_variance", "standard_error", "z_scores")


@pytest.mark.parametrize("window", [7, 31, 65, 201, 1025])
def test_fused_rolling_variance_equals_sort_path_bitwise(window):
    from rocco_b200 import _lib, inference
    lib = _lib.load()
    rng = np.random.default_rng(window)
    m, n = 3, 2 * 131072 + 12345                 # odd n: every other row starts 8 bytes off a 16-byte boundary
    c = rng.normal(size=(m, n)) * (0.2 + np.abs(np.sin(np.arange(n) / 150.0)))
    prev = lib.rocco_b200_trend_set_mode(1)
    try:
        want_s, want = inference._score_centered_wls_matrix(c, prior_df=6.0, spatial_window=window)
    finally:
        lib.rocco_b200_trend_set_mode(0)
    fb0 = lib.rocco_b200_trend_fallback_rows()
    got_s, got = inference._score_centered_wls_matrix(c, prior_df=6.0, spatial_window=window)
    lib.rocco_b200_trend_set_mode(prev)
    assert lib.rocco_b200_trend_fallback_rows() == fb0          # the fused kernel and the multi-select really ran
    assert got["prior_spatial_window"] == window
    assert np.array_equal(got_s, want_s)
    for k in DETAIL_KEYS:
        assert np.array_equal(got[k], want[k]), k
