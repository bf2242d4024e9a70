"""NumPy streams without a GPU: default_rng seeding restated in the library, the checked-in ziggurat tables, and the
argument checks of random_streams."""
import ctypes
import os
import sys

import numpy as np
import pytest

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(REPO, "tools"))

from rocco_b200 import _lib  # noqa: E402

M64 = (1 << 64) - 1
SEEDS = [0, 1, 2**32 - 1, 2**32, 2**64 - 1, 2**64 + 5] + [s + 104729 * (d + 1) for s in (0, 12345, 2**64 - 1) for d in range(25)]


def _state(seed: int):
    out = (ctypes.c_ulonglong * 4)()
    assert _lib.load().rocco_b200_numpy_seed_state(seed & M64, seed >> 64, out) == 0
    return (out[1] << 64) | out[0], (out[3] << 64) | out[2]


@pytest.mark.parametrize("seed", SEEDS)
def test_seed_state_matches_default_rng(seed):
    want = np.random.default_rng(seed).bit_generator.state["state"]
    assert _state(seed) == (want["state"], want["inc"])


def test_tables_match_installed_numpy():
    import gen_numpy_ziggurat as g
    lib = g.default_lib()
    if not os.path.exists(lib):
        pytest.skip("NumPy's libnpyrandom.a is not installed")
    got = g.parse_header(os.path.join(REPO, "rocco_b200", "csrc", "numpy_ziggurat.cuh"))
    want = g.extract(lib)
    assert got["ki"] == want["ki"]
    assert np.array_equal(np.array(got["wi"]).view(np.uint64), np.array(want["wi"]).view(np.uint64))
    assert np.array_equal(np.array(got["fi"]).view(np.uint64), np.array(want["fi"]).view(np.uint64))


def test_budget_params_layout_appends_random_streams():
    prm = _lib.BudgetParams()
    _lib.load().rocco_b200_default_budget_params(ctypes.byref(prm))
    assert prm.random_streams == 0
    names = [f[0] for f in _lib.BudgetParams._fields_]
    assert names[-1] == "random_streams" and names[-2] == "d_innovations"


def test_random_streams_rejections():
    from rocco_b200.inference import random_streams_code
    assert random_streams_code("philox", -3, None) == 0
    assert random_streams_code("numpy", 7, None) == 1
    with pytest.raises(ValueError):
        random_streams_code("pcg", 0, None)
    with pytest.raises(ValueError):
        random_streams_code("numpy", 0, np.zeros(3))
    with pytest.raises(ValueError):
        random_streams_code("numpy", -1, None)


def test_default_flow_args_carry_random_streams():
    from rocco_b200 import pipeline
    assert pipeline.DEFAULT_FLOW_ARGS["random_streams"] == "philox"
    assert pipeline._default_flow_args({"random_streams": "numpy"})["random_streams"] == "numpy"
    with pytest.raises(ValueError):
        pipeline._default_flow_args({"random_streams": "mt19937"})
