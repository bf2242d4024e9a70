"""Column statistics past the per-thread list kernels: the shared-memory tile kernel (k_colstat_tile) against the NumPy /
SciPy oracle at large sample counts, and bit for bit against the list kernels where both run."""
import numpy as np
import pytest

from rocco_b200.synth import chrom_matrix_numpy

pytestmark = pytest.mark.gpu

CENTRAL = (dict(), dict(method="quantile", quantile=0.75), dict(method="quantile", quantile=0.25),
           dict(method="quantile", quantile=0.5, power=2.0), dict(method="mean"), dict(method="t-mean", tprop=0.05),
           dict(method="tmean", tprop=0.2))
DISPERSION = (dict(method="mad"), dict(method="iqr"), dict(method="IQR", rng=(10, 90)), dict(method="std"),
              dict(method="tstd", tprop=0.1))


@pytest.fixture(scope="module")
def lib():
    from rocco_b200 import _lib
    return _lib.load()


@pytest.fixture
def tile_mode(lib):
    """Forces the tile kernel for every m >= 2 while the test runs."""
    prev = lib.rocco_b200_colstat_set_mode(1)
    yield
    lib.rocco_b200_colstat_set_mode(prev)


def _device_stat(x, dtype, kind, kw):
    import torch
    from rocco_b200 import pipeline
    d = torch.from_numpy(np.ascontiguousarray(x, dtype=dtype)).cuda()
    kw = dict(kw)
    if kind == "central":
        kw.setdefault("method", "quantile")
    return pipeline.column_stat_device(d, **kw).cpu().numpy()


def _check(got, want, kind, kw):
    method = kw.get("method", "quantile").lower().replace("-", "")
    exact = (method == "quantile" and kw.get("power", 1.0) == 1.0) or method in ("mean", "mad")
    if exact:
        assert np.array_equal(got, want), kw
    elif kind == "central":
        assert np.allclose(got, want, rtol=1e-13, atol=0), kw
    else:
        assert np.allclose(got, want, rtol=1e-12, atol=1e-300, equal_nan=True), kw


def _signed_ties(m, n, seed):
    """Negative values, heavy ties and both zeros."""
    rng = np.random.default_rng(seed)
    x = np.round(rng.normal(0.0, 2.0, size=(m, n)) * 2.0) / 2.0
    zero = x == 0.0
    x[zero & (rng.random((m, n)) < 0.5)] = -0.0
    x[:, 0] = -0.0
    x[: m // 2, 1] = -0.0
    x[m // 2:, 1] = 0.0
    return x


@pytest.mark.parametrize("m,n", [(769, 300), (1000, 300), (1601, 200), (4096, 120), (16384, 40)])
@pytest.mark.parametrize("data", ["counts", "signed"])
def test_large_m_matches_oracle(oracle, m, n, data):
    x = chrom_matrix_numpy(m, n, seed=m) if data == "counts" else _signed_ties(m, n, seed=m)
    x32 = x.astype(np.float32).astype(np.float64)
    for kind, kws, fn in (("central", CENTRAL, oracle.score_central_tendency_chrom),
                          ("dispersion", DISPERSION, oracle.score_dispersion_chrom)):
        for kw in kws:
            _check(_device_stat(x, np.float64, kind, kw), fn(x, **kw), kind, kw)
            _check(_device_stat(x32, np.float32, kind, kw), fn(x32, **kw), kind, kw)


@pytest.mark.parametrize("m", [2, 3, 10, 11, 100, 129, 300, 768])
@pytest.mark.parametrize("dtype", [np.float64, np.float32])
def test_tile_kernel_equals_list_kernels(lib, m, dtype):
    n = 1_500 if m >= 300 else 5_003
    for x in (chrom_matrix_numpy(m, n, seed=m + 7), _signed_ties(m, n, seed=m + 8)):
        for kind, kws in (("central", CENTRAL), ("dispersion", DISPERSION)):
            for kw in kws:
                prev = lib.rocco_b200_colstat_set_mode(0)
                try:
                    auto = _device_stat(x, dtype, kind, kw)
                    lib.rocco_b200_colstat_set_mode(1)
                    tile = _device_stat(x, dtype, kind, kw)
                finally:
                    lib.rocco_b200_colstat_set_mode(prev)
                assert np.array_equal(auto, tile, equal_nan=True), (m, kind, kw)


def test_public_api_past_768_samples(oracle):
    import rocco_b200
    x = chrom_matrix_numpy(1000, 50_000, seed=11)
    assert np.array_equal(rocco_b200.score_central_tendency_chrom(x, method="mean"),
                          oracle.score_central_tendency_chrom(x, method="mean"))
    assert np.allclose(rocco_b200.score_central_tendency_chrom(x, method="tmean"),
                       oracle.score_central_tendency_chrom(x, method="tmean"), rtol=1e-13, atol=0)


def test_mode_switch_and_sample_limit(lib, tile_mode):
    import torch
    from rocco_b200 import _lib, pipeline
    assert lib.rocco_b200_colstat_set_mode(7) == 1                 # anything but 1 means automatic
    assert lib.rocco_b200_colstat_set_mode(1) == 0
    x = torch.zeros((40_000, 3), dtype=torch.float64, device="cuda")
    x[7] = 2.0
    assert pipeline.column_stat_device(x, "mean").tolist() == [2.0 / 40_000] * 3          # no shared memory: any m
    with pytest.raises(ValueError):
        pipeline.column_stat_device(x, "median")
    assert "at most" in _lib.last_error()
