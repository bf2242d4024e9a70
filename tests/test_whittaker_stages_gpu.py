"""Stage references for the cross-fit Whittaker baseline (csrc/whittaker.cu) over the whole penalty range.

The reference's own float64 solve loses accuracy as the penalty grows (max|oracle64 - b*| ~ 9e-11 at the default window
101, ~5e-7 at window 1001 on the rows below), so the kernels are checked against b*, the same solve carried out in
binary128 and rounded once (``oracle_crossfit_whittaker_baseline_exact``), under

    max|gpu - b*| <= K max|oracle64 - b*| + 1e-13 max|y|

i.e. the GPU is no worse than K times the reference's own error on the same rows.  The tile kernels solve each 9728-bin
tile from a zero state 1280 bins away; that truncation is negligible only while the decay rho of the steady recurrence
keeps rho^1280 <= 1e-12 (windows up to 105).  Larger penalties take the exact sequential path, which must then give the
float64 oracle's bits; ``rocco_b200_whittaker_exact_rows`` tells which path ran.  Penalties below ~10 (window 3, raw
1e-3 and 1) run every tile through the edge kernel: the streaming kernel's right-to-left re-derivation of the forward
solution is unstable there (it was off by 2.7 at lambda = 1e-3).

CPU part (no GPU): b* itself against an exact rational solve and a dense float64 solve, and the float64 oracle against b*.
"""
from fractions import Fraction

import numpy as np
import pytest

# The GPU may be K times the float64 reference's own error.  Measured on a B200, the tile kernels reach 6.6 times it at
# the default penalty, at the last bins of odd-length rows (the edge kernel's tail rows are continued from the steady
# pair, not from the row's own factor); everywhere else they stay below 4 times it.
K = 8.0
FLOOR = 1e-13                 # ... plus this much of max|y|
WT_OUT, HEAD_LEN = 9728, 4096
TILE_WINDOWS = (3, 31, 101, 103, 105)          # rho^1280 <= 1e-12: tile kernels
EXACT_WINDOWS = (107, 109, 151, 201, 301, 1001, 3001)


def _lam(oracle, w):
    return oracle.whittaker_lambda(w)


def _rows(rows, n, seed):
    rng = np.random.default_rng(seed)
    return rng.normal(size=(rows, n)) + 2.0 * np.sin(np.arange(n) / 700.0) + (rng.random((rows, n)) < 0.01) * 6.0


def _gate(err64, y):
    return K * err64 + FLOOR * float(np.max(np.abs(y)))


# ------------------------------------------------------------------ the binary128 reference (CPU)
def _exact_rational(y, lam, parity):
    """W_p + lam D'D solved in rationals (banded Gaussian elimination, no pivoting: the matrix is positive definite)"""
    n = y.size
    lam = Fraction(lam)
    A = [[Fraction(0)] * n for _ in range(n)]
    for i in range(n - 2):                     # D'D from the rows (1, -2, 1) of the second difference
        for a, ca in ((i, 1), (i + 1, -2), (i + 2, 1)):
            for b, cb in ((i, 1), (i + 1, -2), (i + 2, 1)):
                A[a][b] += lam * ca * cb
    rhs = [Fraction(0)] * n
    for i in range(n):
        if i % 2 == parity:
            A[i][i] += 1
            rhs[i] = Fraction(float(y[i]))
    for k in range(n):
        for i in range(k + 1, min(n, k + 3)):
            f = A[i][k] / A[k][k]
            if f:
                for j in range(k, min(n, k + 3)):
                    A[i][j] -= f * A[k][j]
                rhs[i] -= f * rhs[k]
    x = [Fraction(0)] * n
    for i in range(n - 1, -1, -1):
        s = rhs[i] - sum(A[i][j] * x[j] for j in range(i + 1, min(n, i + 3)))
        x[i] = s / A[i][i]
    return x


@pytest.mark.parametrize("n,lam", [(25, 1e-3), (25, 467373.43934201845), (40, 1.0), (40, 4509359321.131039), (31, 1e12)])
def test_binary128_baseline_is_the_rational_solve(oracle, n, lam):
    """b* is the exact solution rounded to double: within one ulp of max|b| of the rational solve, at any penalty"""
    y = _rows(1, n, n)[0]
    xs = [_exact_rational(y, lam, p) for p in (0, 1)]
    want = np.array([float((a + b) / 2) for a, b in zip(*xs)])
    got = oracle.native("port").crossfit_whittaker_baseline_exact(y, lam)
    assert np.max(np.abs(got - want)) <= np.spacing(np.max(np.abs(want))), float(np.max(np.abs(got - want)))


@pytest.mark.parametrize("lam", [1e-3, 0.36, 1.0, 30.0])
def test_binary128_baseline_agrees_with_a_dense_solve(oracle, lam):
    """small lambda, where a dense float64 solve of W_p + lam D'D is accurate to its condition number"""
    n = 64
    y = _rows(1, n, 5)[0]
    D = np.diff(np.eye(n), 2, axis=0)
    fits = []
    for p in (0, 1):
        w = (np.arange(n) % 2 == p).astype(np.float64)
        A = np.diag(w) + lam * (D.T @ D)
        fits.append((np.linalg.solve(A, w * y), np.linalg.cond(A)))
    dense = 0.5 * (fits[0][0] + fits[1][0])
    bound = 8 * n * 2.0 ** -53 * max(c for _, c in fits) * np.max(np.abs(y))
    got = oracle.native("port").crossfit_whittaker_baseline_exact(y, lam)
    assert np.max(np.abs(got - dense)) <= bound, (float(np.max(np.abs(got - dense))), bound)


# the float64 oracle's error against b* on 60000-bin rows (measured: 9.0e-11, 4.5e-10, 1.6e-8, 7.7e-9, 4.1e-7)
@pytest.mark.parametrize("w,err", [(101, 2e-10), (151, 1e-9), (201, 4e-8), (301, 2e-8), (1001, 1e-6)])
def test_float64_oracle_within_its_error(oracle, w, err):
    y = _rows(1, 60000, 1)
    port = oracle.native("port")
    lam = _lam(oracle, w)
    e64 = np.max(np.abs(port.crossfit_whittaker_baseline(y, lam) - port.crossfit_whittaker_baseline_exact(y, lam)))
    assert 0.0 < e64 <= err, e64


# ------------------------------------------------------------------ GPU
@pytest.fixture(scope="module")
def lib():
    from rocco_b200 import _lib
    return _lib.load()


def _check(label, got, y, b64, bstar):
    """per-bin error against b*, and the gate; prints the case's error over the gate for the record"""
    err64 = float(np.max(np.abs(b64 - bstar)))
    gate = _gate(err64, y)
    e = np.abs(got - bstar)
    ratio = float(np.max(e)) / gate
    print(f"WHITTAKER-STAGES {label} gpu_err={float(np.max(e)):.3g} oracle64_err={err64:.3g} gpu/gate={ratio:.3g}")
    return e, gate


def _sweep_lams(oracle):
    out = [(f"w{w}", _lam(oracle, w), False) for w in TILE_WINDOWS]
    out += [(f"w{w}", _lam(oracle, w), True) for w in EXACT_WINDOWS]
    l101 = _lam(oracle, 101)
    out += [("lam1e-3", 1e-3, False), ("lam1", 1.0, False), ("lam101-", l101 * (1 - 1e-9), False),
            ("lam101+", l101 * (1 + 1e-9), False), ("lam1e12", 1e12, True)]
    return out


@pytest.mark.gpu
@pytest.mark.parametrize("n", [60002, 140001])
def test_penalty_sweep(oracle, lib, n):
    """windows 3 ... 3001 and raw penalties 1e-3 ... 1e12 through the drop-in module; the exact path gives the float64
    oracle's bits, the tiles stay within K times its error"""
    from rocco_b200 import _baseline
    port = oracle.native("port")
    y = _rows(3, n, 17 + n)
    failed = []
    for label, lam, exact in _sweep_lams(oracle):
        c0 = lib.rocco_b200_whittaker_exact_rows()
        got = _baseline.crossfit_whittaker_baseline(y, lam)
        took = lib.rocco_b200_whittaker_exact_rows() - c0
        b64 = port.crossfit_whittaker_baseline(y, lam)
        e, gate = _check(f"sweep n={n} {label}", got, y, b64, port.crossfit_whittaker_baseline_exact(y, lam))
        if took != (3 if exact else 0):
            failed.append((label, "exact rows", took))
        if exact and not np.array_equal(got, b64):
            failed.append((label, "bits", int(np.sum(got != b64))))
        if not np.max(e) <= gate:
            failed.append((label, float(np.max(e)), gate))
    assert not failed, failed


def _seams(n):
    """bins around which the kernels change: tile seams, the head-table end, the last two tiles"""
    tiles = (n + WT_OUT - 1) // WT_OUT
    pts = [("seam", t * WT_OUT) for t in range(1, tiles)] + [("head_end", HEAD_LEN)]
    pts += [("tail_tile", max(0, (tiles - 2) * WT_OUT)), ("tail_tile", max(0, (tiles - 1) * WT_OUT)), ("row_end", n - 1)]
    return [(k, p) for k, p in pts if 0 <= p < n]


@pytest.mark.gpu
@pytest.mark.parametrize("w", [101, 301])
@pytest.mark.parametrize("rows,n", [(3, 25), (3, 4104), (3, 4105), (3, 9728), (3, 9729), (3, 11008), (3, 11009),
                                    (3, 12288), (3, 20741), (3, 20742), (24, 300007)])
def test_geometry(oracle, lib, w, rows, n):
    """edge sizes of the head table, the tile and the region, and rows long enough for every persistent cluster to walk
    several tiles; the error profile around every seam is checked against the gate"""
    from rocco_b200 import _baseline
    if w != 101 and rows > 4:
        rows = 4                                  # (exact path: no clusters to exercise, and b* costs CPU time)
    port = oracle.native("port")
    lam = _lam(oracle, w)
    y = _rows(rows, n, 3 * n + w)
    c0 = lib.rocco_b200_whittaker_exact_rows()
    got = _baseline.crossfit_whittaker_baseline(y, lam)
    took = lib.rocco_b200_whittaker_exact_rows() - c0
    b64 = port.crossfit_whittaker_baseline(y, lam)
    e, gate = _check(f"geometry w={w} {rows}x{n}", got, y, b64, port.crossfit_whittaker_baseline_exact(y, lam))
    assert took == (rows if (w > 105 and n > HEAD_LEN + 8) else 0)
    if took:
        assert np.array_equal(got, b64)
    prof = e.max(axis=0)
    for kind, p in _seams(n):
        lo, hi = max(0, p - 64), min(n, p + 64)
        assert prof[lo:hi].max() <= gate, (kind, p, float(prof[lo:hi].max()), gate)
    assert float(np.max(e)) <= gate


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", ["float64", "float32"])
@pytest.mark.parametrize("w", [101, 1001])
def test_fused_scoring_centered_matrix(oracle, lib, w, dtype):
    """log2p1 - row median - baseline as the fused scoring path leaves it, against the same chain with b*; the log2
    may differ by an ulp of its value, once in y and once more through the baseline"""
    import torch
    from rocco_b200 import pipeline
    from rocco_b200.synth import chrom_matrix_numpy
    port = oracle.native("port")
    x = chrom_matrix_numpy(4, 140001, seed=w, dtype=np.float32 if dtype == "float32" else np.float64)
    m = oracle.log_scale_matrix(x.astype(np.float64))
    g = m - np.median(m, axis=1, keepdims=True)
    lam = _lam(oracle, w)
    c0 = lib.rocco_b200_whittaker_exact_rows()
    _, det = pipeline.score_loci_wls_device(torch.from_numpy(x).cuda(), details=True,
                                            params=pipeline.score_params(baseline_window=w, exact_pilot=True))
    took = lib.rocco_b200_whittaker_exact_rows() - c0
    assert det["local_baseline_window"] == w and det["local_baseline_lambda"] == lam
    assert took == (4 if w > 105 else 0)
    got = det["centered_matrix"].cpu().numpy()
    bstar = port.crossfit_whittaker_baseline_exact(g, lam)
    e, gate = _check(f"fused w={w} {dtype}", g - got, g, port.crossfit_whittaker_baseline(g, lam), bstar)
    gate += 2.0 * float(np.spacing(np.max(np.abs(m))))
    assert float(np.max(e)) <= gate, (float(np.max(e)), gate)


@pytest.mark.gpu
def test_local_background_window_301(oracle, lib):
    from rocco_b200 import inference
    port = oracle.native("port")
    y = _rows(3, 60002, 301)
    c0 = lib.rocco_b200_whittaker_exact_rows()
    base, w, lam = inference._estimate_local_background_matrix(y, target_window=301)
    assert (w, lam) == (301, _lam(oracle, 301))
    assert lib.rocco_b200_whittaker_exact_rows() - c0 == 3
    b64 = port.crossfit_whittaker_baseline(y, lam)
    assert np.array_equal(base, b64)
    e, gate = _check("local_background w=301", base, y, b64, port.crossfit_whittaker_baseline_exact(y, lam))
    assert float(np.max(e)) <= gate
