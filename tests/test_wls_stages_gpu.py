"""Stage-level references for the WLS variance chain: the rolling AR(1) variance, the trend's order statistics, PAVA and
knot interpolation, and the combine across the knot-table batches, each against a plain high-precision restatement of the
same operation rather than against another GPU kernel.

With one sample row, ``raw_variance`` is ``1 / rcp(V)`` and ``prior_variance`` is ``1 / rcp(trend)`` (wls.cu, k_combine):
both are within a couple of ulps of the row's own V and trend while V < 1e8, so the per-row stages are observed through the
public API.

A. Rolling variance.  Test rows are put on a grid of 2^-35, so every window's sums s1, s2 and sl are exact integers
   (int64 prefix sums of the value split into two 25-bit halves); the reference formula (oracle_wls.c:206-236) is then
   applied in long double.  Its error is ~2^-62 of the window's sum of squares, 2^-14 of the bound below.
   Bound for output j, from the kernels' summation (a w-term direct sum for the first output of every block of 8, then
   at most 7 slides), the cancellation in g0 and g1, beta's amplification (den >= g0 c1, the clamp is 1-Lipschitz) and
   the m = 1 reciprocal round trip:
       |V_gpu - V_true| <= 32 (w + 16) u S2x_j / w + 4 u V_true,    u = 2^-53.
   S2x_j is the sum of squares of every element the sums of that window touched: the window and the up to 7 elements that
   slid out of it since the block's direct sum.  With the window's own sum of squares instead, the bound does not hold
   after a downward scale step (1 -> 2^-12, 2^11 -> 1): an element that slid out leaves the rounding of its square in s2.
   Measured on a B200, the error reaches 1.7e3 times that variant of the bound at w = 31 (``own_s2`` in the printed
   report) and 0.014 times the bound above.
B. Trend.  The oracle's fit_variance_trend is fed the GPU's own V (recovered from raw_variance), so the comparison
   isolates the order statistics, PAVA, knot de-duplication, the knot table and its LUT walk from the variance rounding.
   Bound: 32 u max(|y_lo|, |y_hi|) of the knot segment + 4 u trend (round trip).  An order statistic one rank off moves a
   knot by ~1/n relative, about 10^7 times this.
C. Combine.  Each row's V and trend come from its own one-row call; the m-row outputs are recomputed from them with
   math.fsum (oracle_wls.c:281-304) within 8 (m + 8) u of the sum of absolute terms.
"""
import math

import numpy as np
import pytest

from tests.conftest import rel_err

U = 2.0 ** -53
TOL, TIGHT = 1e-5, 1e-6            # the project's gate and its regression guard (test_score_gpu.py)
RV_T, RV_CHUNK = 4096, 61440        # fused rolling-variance tile and CTA chunk (trend.cu)
QBITS = 35                          # test rows live on a grid of 2^-35 (|c| < 2^15): exact integer window sums
DETAIL_KEYS = ("mean", "raw_variance", "prior_variance", "moderated_variance", "standard_error", "z_scores")
FB_NAMES = {1: "xslot", 2: "xcount", 4: "ytotal", 8: "yslot", 16: "ycount"}


def resolve_window(n, requested):
    """wls_backend.c:232-260"""
    if n < 5:
        return 0
    w = requested if requested > 0 else 31
    w = max(w, 5)
    w = min(w, n)
    if w % 2 == 0:
        w = w - 1 if w == n else w + 1
    return w if w >= 5 else 0


# ------------------------------------------------------------------ A: the reference
class _ExactSums:
    """Exact window sums of a row on the 2^-QBITS grid: a = c 2^QBITS = ah 2^25 + al (0 <= al < 2^25, |a| < 2^50), so
    every product of halves is < 2^50 and a window of up to 4097 of them fits int64.  Prefix sums wrap modulo 2^64;
    differences of them are exact because the window sums fit."""

    def __init__(self, c):
        a = np.rint(np.ldexp(c, QBITS))
        assert np.array_equal(np.ldexp(a, -QBITS), c) and np.max(np.abs(a), initial=0.0) < 2.0 ** 50, "row is not on the grid"
        a = a.astype(np.int64)
        self.a = a
        ah, al = a >> 25, a & ((1 << 25) - 1)
        with np.errstate(over="ignore"):
            def pre(x):
                return np.concatenate(([0], np.cumsum(x, dtype=np.int64)))
            self.p1 = pre(a)
            self.p2 = [pre(ah * ah), pre(ah * al), pre(al * al)]
            self.pl = [pre(ah[:-1] * ah[1:]), pre(ah[:-1] * al[1:]), pre(al[:-1] * ah[1:]), pre(al[:-1] * al[1:])]

    @staticmethod
    def _d(p, lo, hi):
        with np.errstate(over="ignore"):
            return (p[hi] - p[lo]).astype(np.longdouble)

    def s1(self, lo, hi):
        return self._d(self.p1, lo, hi)

    def s2(self, lo, hi):
        hh, hl, ll = (self._d(p, lo, hi) for p in self.p2)
        return np.ldexp(hh, 50) + np.ldexp(hl, 26) + ll

    def sl(self, lo, hi):                 # sum of a_k a_{k+1} for k in [lo, hi - 1)
        hh, hl, lh, ll = (self._d(p, lo, hi - 1) for p in self.pl)
        return np.ldexp(hh, 50) + np.ldexp(hl + lh, 25) + ll


def ar1_reference(c, window):
    """(V_true, S2x, S2_own) per output of one row: the rolling AR(1) innovation variance of oracle_wls.c:188-239 from
    exact window sums in long double, floored at 1e-8 like the kernels (wls_backend.c:869); S2x and S2_own as in the
    module docstring.  Returns None where the row takes the constant path (no window)."""
    c = np.ascontiguousarray(c, dtype=np.float64)
    n = c.shape[0]
    w = resolve_window(n, window)
    if w == 0 or n < 4:
        return None
    E = _ExactSums(c)
    half, last = w // 2, n - w
    t = np.arange(last + 1)
    ld = np.longdouble
    sc2 = ld(2.0) ** (-2 * QBITS)
    s1, s2, sl = E.s1(t, t + w), E.s2(t, t + w), E.sl(t, t + w)
    first, lastv = E.a[t].astype(ld), E.a[t + w - 1].astype(ld)
    wd = ld(w)
    # integer units: g0 w = s2 w - s1^2 ; g1 w^2 = sl w^2 - s1 w (2 s1 - first - last) + (w - 1) s1^2
    g0 = (s2 * wd - s1 * s1) / wd * sc2
    g1 = (sl * wd * wd - s1 * wd * (2 * s1 - first - lastv) + (wd - 1) * s1 * s1) / (wd * wd) * sc2
    g0 = np.maximum(g0, ld(0))
    shrink = ld(1) / (wd + ld(1))
    den = g0 * (ld(1) + shrink) + ld(1.0e-4) * (g0 + ld(1))
    eps = ld(1.0e-12) * (g0 + ld(1))
    beta = np.where(den > eps, g1 / den, ld(0))
    beta = np.clip(beta, ld(0), ld(0.99))
    omb = np.maximum(ld(1) - beta * beta, ld(0))
    at_start = np.maximum(g0 / wd * omb, ld(0))
    j = np.arange(n)
    tj = np.clip(j - half, 0, last)
    v = np.maximum(at_start[tj], ld(1.0e-8))
    s2x = (E.s2(np.maximum(tj - 7, 0), tj + w) * sc2).astype(np.float64)
    s2o = (E.s2(tj, tj + w) * sc2).astype(np.float64)
    return v, s2x, s2o


def ar1_bound(v_true, s2, w):
    return 32.0 * (w + 16) * U * s2 / w + 4.0 * U * np.asarray(v_true, dtype=np.float64)


# ------------------------------------------------------------------ A: the data
def _ar1(rng, length, phi, scale=1.0):
    if phi == 0.0:
        return rng.standard_normal(length) * scale
    from scipy.signal import lfilter
    e = rng.standard_normal(length) * math.sqrt(1.0 - phi * phi)
    x = lfilter([1.0], [1.0, -phi], e, zi=[phi * rng.standard_normal()])[0]
    return x * scale


def a_row(n, seed, down_jumps=False):
    """Segments on tile seams (2048 bins for rows of three tiles or more, else n // 7): AR(1) with phi in {0, 0.5, 0.9,
    0.98, 0.999} (the 0.999 segments carry a smooth peak, so beta reaches the 0.99 clamp where w > 98; below that
    den >= g0 (1 + 1/(w+1)) and g1 <= g0 keep beta under it), offsets of 3-10 sigma over a few hundred bins (large mu),
    runs of exact zeros (V on the 1e-8 floor), all on the 2^-35 grid.  Rows of ten segments or more also jump in scale:
    a 2^-12 segment first and a 2^11 segment last (up-jumps only), or with `down_jumps` the 2^-12 segment after unit-scale
    ones and the 2^11 segment in the middle.  A down-jump is where the reference's whole-row slide fails the 1e-6 gate by
    itself: the rounding of the large squares it slid over stays in its sums (up to 1e-5 relative on the small segment),
    so rows with down-jumps are checked against the exact reference only."""
    rng = np.random.default_rng(seed)
    seg = 2048 if n >= 3 * RV_T else max(4, n // 7)
    bounds = list(range(0, n, seg)) + [n]
    nseg = len(bounds) - 1
    cycle = [("ar", 0.0), ("ar", 0.5), ("ar", 0.9), ("ar", 0.98), ("ar", 0.999), ("offsets", 0.5), ("zeros", 0.0)]
    out = np.empty(n)
    for i in range(nseg):
        s, e = bounds[i], bounds[i + 1]
        L = e - s
        kind, phi = cycle[i % len(cycle)]
        scale = 1.0
        if nseg >= 10 and i == (7 if down_jumps else 0):
            kind, phi, scale = "ar", 0.9, 2.0 ** -12
        elif nseg >= 10 and i == (nseg // 2 if down_jumps else nseg - 1):
            kind, phi, scale = "ar", 0.0, 2.0 ** 11
        if kind == "zeros":
            out[s:e] = 0.0
        elif kind == "offsets":
            x = _ar1(rng, L, phi)
            p = 0
            while p < L:
                q = min(L, p + int(rng.integers(150, 400)))
                x[p:q] += rng.uniform(3.0, 10.0) * rng.choice([-1.0, 1.0])
                p = q
            out[s:e] = x
        else:
            out[s:e] = _ar1(rng, L, phi, scale)
            if phi == 0.999:                              # a smooth peak: beta reaches the clamp (w > 98 only)
                wd = min(L, 400)
                p0 = s + (L - wd) // 2
                out[p0:p0 + wd] += 8.0 * np.sin(np.pi * (np.arange(wd) + 0.5) / wd)
    out = np.clip(out, -30000.0, 30000.0)
    return np.ldexp(np.rint(np.ldexp(out, QBITS)), -QBITS)


# ------------------------------------------------------------------ A: CPU check of the reference itself
@pytest.mark.parametrize("n,window", [(5, 31), (6, 8), (7, 7), (9, 10), (12, 12), (13, 64), (16, 6), (21, 200), (33, 34),
                                      (40, 40), (40, 39), (64, 31), (300, 5), (700, 65), (1500, 201), (2100, 1025)])
def test_ar1_reference_matches_oracle_on_short_rows(oracle, n, window):
    """the long-double reference against the oracle's own sliding restatement; on short unit-scale rows the oracle's
    drift (every slide since the row's start) is tiny, so the bound carries the whole prefix's sum of squares"""
    c = a_row(n, seed=n * 7 + window)
    w = resolve_window(n, window)
    got = oracle.native("port").rolling_ar1_variance(c, window)
    v, _, _ = ar1_reference(c, window)
    half, last = w // 2, n - w
    tj = np.clip(np.arange(n) - half, 0, last)
    pre = np.concatenate(([0.0], np.cumsum(c * c)))
    s2_prefix = pre[tj + w] * (1 + 1e-12)
    want = np.asarray(v, dtype=np.float64)
    got = np.maximum(got, 1.0e-8)
    bound = 32.0 * (w + 16 + tj) * U * s2_prefix / w + 4.0 * U * want
    assert np.all(np.abs(got - want) <= bound), float(np.max(np.abs(got - want) / bound))


def test_ar1_reference_resolves_windows_like_the_oracle(oracle):
    for n in range(1, 41):
        for req in (-3, 0, 4, 5, 6, 7, 8, n - 1, n, n + 1, 2 * n, 31, 1000):
            assert resolve_window(n, req) == oracle.native("port").score_centered_wls(
                np.ones((1, n)), spatial_window=req)[7], (n, req)


def test_a_rows_hit_the_clamp_the_floor_and_large_means():
    """the data reach what the issue's gaps name: beta at the 0.99 clamp, V on the 1e-8 floor, |mu| of several sigma"""
    n, w = 2 * RV_CHUNK + 1, 201
    c = a_row(n, seed=1)
    v, s2x, _ = ar1_reference(c, w)
    assert np.any(np.asarray(v, dtype=np.float64) == 1.0e-8)
    mu = np.convolve(c, np.ones(w) / w, mode="valid")
    assert np.max(np.abs(mu)) > 3.0
    # the clamp: some window's beta reaches 0.99 (recompute it from the float sums, plenty for this)
    E = _ExactSums(c)
    t = np.arange(n - w + 1)
    s1 = np.asarray(E.s1(t, t + w), dtype=np.float64) * 2.0 ** -QBITS
    s2 = np.asarray(E.s2(t, t + w), dtype=np.float64) * 2.0 ** (-2 * QBITS)
    sl = np.asarray(E.sl(t, t + w), dtype=np.float64) * 2.0 ** (-2 * QBITS)
    m = s1 / w
    g0 = s2 - w * m * m
    g1 = sl - m * (2 * s1 - c[t] - c[t + w - 1]) + (w - 1) * m * m
    beta = g1 / (g0 * (1 + 1 / (w + 1)) + 1e-4 * (g0 + 1))
    assert np.any(beta > 0.99) and np.any(beta < 0.0)


# ------------------------------------------------------------------ GPU plumbing
def _lib():
    from rocco_b200 import _lib as L
    return L.load()


def _fb_reasons(lib):
    import ctypes
    buf = (ctypes.c_longlong * 8)()
    lib.rocco_b200_trend_fallback_reasons(ctypes.cast(buf, ctypes.c_void_p))
    return np.array(list(buf), dtype=np.int64)


def _gpu(c, mode, **kw):
    """scores, details, fallback rows and fallback reasons this call added, in trend mode `mode`"""
    from rocco_b200 import inference
    lib = _lib()
    prev = lib.rocco_b200_trend_set_mode(mode)
    try:
        fb0, r0 = lib.rocco_b200_trend_fallback_rows(), _fb_reasons(lib)
        sc, det = inference._score_centered_wls_matrix(np.ascontiguousarray(c, dtype=np.float64), **kw)
        fb, rs = lib.rocco_b200_trend_fallback_rows() - fb0, _fb_reasons(lib) - r0
    finally:
        lib.rocco_b200_trend_set_mode(prev)
    return sc, det, int(fb), rs


def _reason_text(rs):
    return ",".join(f"{FB_NAMES[1 << k]}:{int(rs[k])}" for k in range(5) if rs[k]) or "-"


# ------------------------------------------------------------------ A on the GPU
def _a_lengths(w):
    h = w // 2
    out = [w, w + 1, w + 7]
    for base in (2 * RV_CHUNK, 3 * RV_T):
        out += [base - 1, base + 1, base - h, base + h]
    return sorted(set(out))


A_WINDOWS = (5, 7, 31, 33, 65, 201, 1023, 1025, 1027, 2049, 4097)
A_CASES = [(w, n) for w in A_WINDOWS for n in _a_lengths(w)]
A_SMALL = [(5, 31), (6, 31), (7, 8), (9, 10), (12, 12), (13, 64), (16, 6), (21, 200), (33, 34), (40, 40), (40, 39),
           (11, 4), (25, 26)]


def _check_a(c, window, label, gate=True, score_tol=TIGHT):
    m, n = c.shape
    w = resolve_window(n, window)
    refs = [ar1_reference(c[r], window) for r in range(m)]
    if gate:
        from oracle import oracle as orc
        want_s, want = orc.score_centered_wls_matrix(c, spatial_window=window)
    worst, worst_own = 0.0, 0.0
    for mode in (0, 1):
        sc, det, fb, rs = _gpu(c, mode, spatial_window=window)
        assert det["prior_spatial_window"] == w
        raw = det["raw_variance"]
        if m == 1:
            v, s2x, s2o = refs[0]
            vt = np.asarray(v, dtype=np.float64)
            err = np.abs(raw - vt)
            ratio = err / ar1_bound(vt, s2x, w)
            own = err / ar1_bound(vt, s2o, w)
        else:
            # harmonic mean H = m / sum(1/V_r): dH = sum_r H^2 / (m V_r^2) dV_r, plus the rounding of the sum itself
            vts = [np.asarray(r[0], dtype=np.float64) for r in refs]
            inv = np.sum([1.0 / x for x in vts], axis=0)
            H = m / inv
            b = sum(H * H / (m * x * x) * ar1_bound(x, r[1], w) for x, r in zip(vts, refs)) + 4.0 * (m + 2) * U * H
            bo = sum(H * H / (m * x * x) * ar1_bound(x, r[2], w) for x, r in zip(vts, refs)) + 4.0 * (m + 2) * U * H
            err = np.abs(raw - H)
            ratio, own = err / b, err / bo
        worst = max(worst, float(np.max(ratio)))
        worst_own = max(worst_own, float(np.max(own)))
        assert np.all(ratio <= 1.0), (label, mode, int(np.argmax(ratio)), float(np.max(ratio)))
        if not gate:
            continue
        e = rel_err(sc, want_s)
        assert e <= score_tol, (label, mode, "scores", e)
        for k in DETAIL_KEYS:
            e = rel_err(det[k], want[k])
            assert e <= (score_tol if k == "z_scores" else TIGHT), (label, mode, k, e)
    print(f"WLS-STAGES A {label} w={w} m={m} n={n} max_err/bound={worst:.3g} own_s2={worst_own:.3g}")
    return worst


@pytest.mark.gpu
@pytest.mark.parametrize("window,n", A_CASES)
def test_rolling_variance_against_exact_reference(window, n):
    c = a_row(n, seed=window * 1000003 + n)[None, :]
    _check_a(c, window, f"w{window}_n{n}")


@pytest.mark.gpu
@pytest.mark.parametrize("window", [5, 31, 201, 1025, 2049])
def test_rolling_variance_after_scale_down_jumps(window):
    """1 -> 2^-12 and 2^11 -> 1 steps: the windows after them carry the rounding of squares that slid out, which the
    bound's S2x covers and the window's own sum of squares does not (own_s2 in the report)"""
    n = 2 * RV_CHUNK + 1
    c = a_row(n, seed=window * 17 + 3, down_jumps=True)[None, :]
    _check_a(c, window, f"down_w{window}", gate=False)


@pytest.mark.gpu
@pytest.mark.parametrize("window", A_WINDOWS)
def test_rolling_variance_three_rows_odd_length(window):
    """m = 3 with odd n: rows start in both 16-byte alignment classes; the harmonic mean against the per-row truths.
    Scores and z are held to the 1e-5 gate here, the details to 1e-6: where the rows' values cancel in the weighted mean,
    the reference's own slide drift (V ~3e-8 relative) reaches the scores -- at w = 201 the oracle's scores differ by
    1.3e-6 from the same combine fed the exact V, and the GPU's by the same amount from the oracle."""
    n = 2 * 131072 + 12345
    c = np.stack([a_row(n, seed=window * 31 + r) for r in range(3)])
    _check_a(c, window, f"w{window}_m3", score_tol=TOL)


@pytest.mark.gpu
@pytest.mark.parametrize("n,window", A_SMALL)
def test_rolling_variance_small_rows_resolve_the_window(n, window):
    c = a_row(n, seed=n * 100 + window)[None, :]
    _check_a(c, window, f"small_n{n}_req{window}")


# ------------------------------------------------------------------ B: trend against the oracle fed the GPU's own V
def b_row(n, seed, k=0, peak=32.0, peak_frac=0.036, low_frac=0.04, sigma=0.2):
    """One row family: background noise; 200-bin peak segments (sigma x `peak`) and low segments (sigma / 32), so that the
    variances spread 2^+-10 around the median; the 1500 |C| values nearest every bin-boundary quantile set to it exactly
    (thousands of ties where the bins are cut); scaled by 2^k (exact)."""
    rng = np.random.default_rng(seed)
    c = rng.standard_normal(n) * sigma * (1.0 + 0.5 * np.sin(np.arange(n) / 150.0))
    for frac, f in ((peak_frac, peak), (low_frac, 1.0 / 32.0)):
        for s in rng.choice(n // 200, size=int(frac * n / 200), replace=False) * 200:
            c[s:s + 200] *= f
    B = int(max(4.0, math.floor(1.0 + math.log(n + 1.0) / math.log(2.0))))
    a = np.abs(c)
    order = np.argsort(a, kind="stable")
    for b in range(1, B):
        r = (b * n) // B
        sel = order[max(0, r - 750): r + 750]
        c[sel] = np.where(c[sel] < 0, -1.0, 1.0) * a[order[r]]
    return np.ldexp(c, k)


def one_knot_row(n, seed):
    """every |C| but twenty is 0.5 (random signs): every bin's x-median is equal, so the trend is one knot"""
    rng = np.random.default_rng(seed)
    c = rng.choice([-0.5, 0.5], size=n)
    c[rng.choice(n, 20, replace=False)] = rng.standard_normal(20)
    return c


def _trend_bound(c, want, kx, ky):
    t = np.abs(c)
    if kx.size >= 2:
        i = np.clip(np.searchsorted(kx, t, side="right") - 1, 0, kx.size - 2)
        scale = np.maximum(np.abs(ky[i]), np.abs(ky[i + 1]))
    else:
        scale = np.abs(want)
    return 32.0 * U * scale + 4.0 * U * np.abs(want)


# (label, row builder, designed path of mode 0: "fast" = no fallback, else the fallback reason expected)
B_CASES = [
    *[(f"scale2^{k}", (lambda k=k: b_row(200_003, 40 + k, k)), "xslot" if k in (-20, 8) else "fast") for k in (-20, -12, -6, 0, 4, 8)],
    ("one_knot_6000", lambda: one_knot_row(6000, 3), "fast"),
    ("one_knot_200003", lambda: one_knot_row(200_003, 4), "xslot"),
    ("rows_6M", lambda: b_row(6_000_000, 6, 0, peak=8.0, peak_frac=0.01, low_frac=0.01), "fast"),
    ("large_12.5M", lambda: b_row(12_500_000, 12, 0, peak=10.0, peak_frac=0.01, low_frac=0.01, sigma=0.25), "fast"),
    ("large_12.5M_dense_peaks", lambda: b_row(12_500_000, 13, 0, peak=10.0, peak_frac=0.08, low_frac=0.01, sigma=0.25), "yslot"),
]


@pytest.mark.gpu
@pytest.mark.parametrize("label,make,path", B_CASES, ids=[c[0] for c in B_CASES])
def test_trend_against_oracle_fed_gpu_variance(oracle, label, make, path):
    c = make()
    port = oracle.native("port")
    worst = 0.0
    for mode in (0, 1):
        sc, det, fb, rs = _gpu(c[None, :], mode)
        v_gpu = det["raw_variance"]
        assert np.max(v_gpu) < 1e8                              # the reciprocal round trip holds below 1e8
        want, kx, ky = port.fit_variance_trend(c, v_gpu)
        want = np.maximum(want, 1.0e-8)
        got = det["prior_variance"]
        ratio = np.abs(got - want) / _trend_bound(c, want, kx, ky)
        worst = max(worst, float(np.max(ratio)))
        assert np.all(ratio <= 1.0), (label, mode, int(np.argmax(ratio)), float(np.max(ratio)))
        if mode == 0:
            taken = "fast" if fb == 0 else _reason_text(rs)
            print(f"WLS-STAGES B {label} n={c.size} knots={kx.size} path={taken} max_err/bound=", end="")
            if path == "fast":
                assert fb == 0, (label, _reason_text(rs))
            else:
                bit = next(k for k, v in FB_NAMES.items() if v == path).bit_length() - 1
                assert fb == 1 and rs[bit] == 1, (label, _reason_text(rs))
    print(f"{worst:.3g}")


# ------------------------------------------------------------------ C: combine across the knot-table batches
C_N = 3001
C_MAX_M = 83


@pytest.fixture(scope="module")
def c_rows():
    """83 rows, row r scaled by 2^((r mod 9) - 4), with each row's V and trend from its own one-row call"""
    rng = np.random.default_rng(2024)
    rows = np.empty((C_MAX_M, C_N))
    for r in range(C_MAX_M):
        rows[r] = b_row(C_N, 500 + r, 0, peak=8.0, peak_frac=0.1, low_frac=0.05) * 2.0 ** ((r % 9) - 4) \
            + rng.normal() * 0.05
    per_row = []
    for r in range(C_MAX_M):
        _, det, _, _ = _gpu(rows[r:r + 1], 0, prior_df=6.0)
        per_row.append((det["raw_variance"], det["prior_variance"]))
    return rows, per_row


def combine_reference(y, V, T, ldf, pdf, pfr, lower_bound_z=1.0, min_effect=None):
    """oracle_wls.c:281-304 per bin with exact sums (math.fsum); returns the outputs and their error bounds"""
    m, n = y.shape
    tdf = ldf + pdf
    ov, pv = np.maximum(V, 1e-8), np.maximum(T, 1e-8)
    post = (ldf * ov + pdf * pv) / max(tdf, 1.0)
    post = np.maximum(np.maximum(post, pfr * pv), 1e-8)
    prec = 1.0 / post
    fs = lambda a: np.array([math.fsum(a[:, j]) for j in range(n)])     # noqa: E731
    psum, wsum, rsum, qsum = fs(prec), fs(prec * y), fs(1.0 / ov), fs(1.0 / pv)
    wabs = fs(np.abs(prec * y))
    P = np.maximum(psum, 1e-8)
    mean = wsum / P
    se = np.sqrt(1.0 / P)
    out = {"mean": mean, "raw_variance": m / np.maximum(rsum, 1e-8), "prior_variance": m / np.maximum(qsum, 1e-8),
           "moderated_variance": m / P, "standard_error": se}
    z = mean / np.maximum(se, 1e-8)
    me = None if min_effect is None else max(min_effect, 0.0)
    score = z - lower_bound_z if me is None else (mean - me) / np.maximum(se, 1e-8)
    out["z_scores"] = z
    g = 8.0 * (m + 8) * U
    dmean = g * (wabs + np.abs(mean) * psum) / P
    bnd = {"mean": dmean, "raw_variance": g * out["raw_variance"], "prior_variance": g * out["prior_variance"],
           "moderated_variance": g * out["moderated_variance"], "standard_error": g * se}
    bnd["z_scores"] = dmean / se + np.abs(z) * g + g * np.abs(z)
    shift = abs(lower_bound_z) if me is None else me / np.maximum(se, 1e-8)       # rounding of the subtraction
    bnd["scores"] = dmean / se + 2.0 * g * np.abs(score) + g * shift
    return score, out, bnd


def _check_combine(y, V, T, label, w_resolved, **kw):
    m = y.shape[0]
    ldf = max(4.0, w_resolved - 3.0) if w_resolved > 0 else 1.0
    pdf = max(kw.get("prior_df", 5.0), 0.0)
    pfr = max(kw.get("precision_floor_ratio", 0.01), 0.0)
    score, want, bnd = combine_reference(y, V, T, ldf, pdf, pfr, kw.get("lower_bound_z", 1.0), kw.get("min_effect"))
    sc, det, _, _ = _gpu(y, 0, **kw)
    worst = float(np.max(np.abs(sc - score) / bnd["scores"]))
    assert worst <= 1.0, (label, "scores", worst)
    for k in DETAIL_KEYS:
        r = float(np.max(np.abs(det[k] - want[k]) / bnd[k]))
        assert r <= 1.0, (label, k, r)
        worst = max(worst, r)
    print(f"WLS-STAGES C {label} m={m} max_err/bound={worst:.3g}")


@pytest.mark.gpu
@pytest.mark.parametrize("m", [1, 4, 5, 39, 40, 41, 44, 45, 83])
def test_combine_across_knot_table_batches(c_rows, m):
    rows, per_row = c_rows
    V = np.stack([per_row[r][0] for r in range(m)])
    T = np.stack([per_row[r][1] for r in range(m)])
    _check_combine(rows[:m], V, T, f"m{m}", 31, prior_df=6.0)


@pytest.mark.gpu
@pytest.mark.parametrize("kw", [dict(prior_df=0.0), dict(prior_df=6.0, precision_floor_ratio=0.5),
                                dict(prior_df=6.0, min_effect=0.3), dict(prior_df=6.0, lower_bound_z=0.0)],
                         ids=["prior_df0", "floor0.5", "min_effect", "lbz0"])
def test_combine_parameters_at_41_rows(c_rows, kw):
    rows, _ = c_rows
    m = 41
    per = [_gpu(rows[r:r + 1], 0, **kw)[1] for r in range(m)]
    V = np.stack([d["raw_variance"] for d in per])
    T = np.stack([d["prior_variance"] for d in per])
    if "precision_floor_ratio" in kw:
        post = (28.0 * V + 6.0 * T) / 34.0
        assert np.mean(post < 0.5 * T) > 0.05                  # the floor binds on part of the bins
    _check_combine(rows[:m], V, T, "m41_" + "_".join(kw), 31, **kw)


@pytest.mark.gpu
@pytest.mark.parametrize("n", [1, 2, 3, 4])
def test_combine_constant_rows_at_41_rows(oracle, n):
    """n <= 4: no window, each row's variance is its robust scale squared (k_robust_rows) on both tracks"""
    rng = np.random.default_rng(n)
    m = 41
    y = rng.standard_normal((m, n)) * (2.0 ** ((np.arange(m) % 9) - 4))[:, None]
    per = [_gpu(y[r:r + 1], 0, prior_df=6.0)[1] for r in range(m)]
    V = np.stack([d["raw_variance"] for d in per])
    T = np.stack([d["prior_variance"] for d in per])
    assert np.array_equal(V, T)
    for r in range(m):                                          # robust scale^2 of the row (oracle_wls.c:58-67)
        med = np.median(y[r])
        sc = max(np.median(np.abs(y[r] - med)) * 1.4826, 1e-6)
        assert abs(V[r, 0] - max(sc * sc, 1e-8)) <= 4 * U * V[r, 0]
    _check_combine(y, V, T, f"const_n{n}", 0, prior_df=6.0)
    want_s, want = oracle.score_centered_wls_matrix(y, prior_df=6.0)
    got_s, got = _gpu(y, 0, prior_df=6.0)[:2]
    assert rel_err(got_s, want_s) <= TIGHT
