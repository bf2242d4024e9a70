// EB-moderated WLS locus scoring on a centered matrix, and the score_loci_wls chain around it.
//
// Replaces /root/reference/rocco/native/wls_backend.c:
//   610-742  rolling AR(1) innovation variance   -> k_rollvar   (direct window sums + short slides)
//   394-608  monotone variance-vs-|signal| trend -> exact order statistics per sample row, PAVA on <= 32 knots
//   744-947  posterior precision + combine       -> k_combine   (fused column reduction over the sample axis)
// and the Python driver inference.py:302-379.
#include <stdlib.h>

#include <condition_variable>
#include <deque>
#include <mutex>
#include <thread>

#include "common.cuh"
#include "select.cuh"
#include "score.cuh"
#include "trend.cuh"

#include <cub/cub.cuh>
#include <math.h>

#include <algorithm>

namespace rb {
namespace score {

int resolve_spatial_window(long long n, int requested)          // wls_backend.c:232-260
{
    if (n < 5) return 0;
    long long w = requested > 0 ? requested : 31;
    if (w < 5) w = 5;
    if (w > n) w = n;
    if ((w & 1) == 0) w = (w == n) ? (w - 1) : (w + 1);
    return (w < 5) ? 0 : (int)w;
}

int resolve_baseline_window(long long n, int target)             // inference.py:50-62
{
    if (n < 25) return 0;
    long long w = std::max(3, target);
    if (w > n) w = n;
    if ((w % 2) == 0) w = (w == n) ? w - 1 : w + 1;
    return (int)std::max<long long>(0, w);
}

double whittaker_lambda(int block)                                // inference.py:65-76
{
    int b = std::max(3, block);
    if ((b % 2) == 0) b += 1;
    const double w_hat = (double)b * 0.15915494;
    return 7.0 * pow(w_hat, 4.0);                                 // CPython float ** 4 is libm pow
}

// ------------------------------------------------------------------ small helpers
__device__ __forceinline__ double load_logx(const void *x, int in_f32, long long idx)
{
    const double v = in_f32 ? (double)reinterpret_cast<const float *>(x)[idx] : reinterpret_cast<const double *>(x)[idx];
    return log2(fmax(v, 0.0) + 1.0);
}

constexpr int PILOT_CAP = 4096;

// inference.py:333  np.median(matrix, axis=1): exact for n <= 4096, sampled above (see score.cuh)
__global__ void __launch_bounds__(256) k_pilot(const void *x, int in_f32, long long n, long long row_stride, double *pilot)
{
    // the values are log2(max(x, 0) + 1) >= 0 (NaN -> +inf): their bit patterns order like the values, so the one or two
    // middle ranks come from a radix select instead of a sort
    __shared__ unsigned long long s[PILOT_CAP];
    __shared__ SelScratch S;
    const long long row = blockIdx.x;
    const int take = (int)min((long long)PILOT_CAP, n);
    for (int k = threadIdx.x; k < take; k += 256) {
        const long long i = (n <= PILOT_CAP) ? k : (long long)(((double)k + 0.5) * ((double)n / (double)PILOT_CAP));
        double v = load_logx(x, in_f32, row * row_stride + min(i, n - 1));
        if (!(v == v)) v = INFINITY;
        s[k] = (unsigned long long)__double_as_longlong(v);
    }
    __syncthreads();
    const double hi = __longlong_as_double((long long)block_select<256>(s, take, take / 2, nullptr, 0ULL, S, nullptr, nullptr));
    double lo = hi;
    if (!(take & 1)) lo = __longlong_as_double((long long)block_select<256>(s, take, take / 2 - 1, nullptr, 0ULL, S, nullptr, nullptr));
    if (threadIdx.x == 0) pilot[row] = (take & 1) ? hi : (lo + hi) / 2.0;
}

__global__ void k_pilot_keys(const void *x, int in_f32, long long n, long long base, unsigned long long *keys)
{
    for (long long j = (long long)blockIdx.x * blockDim.x + threadIdx.x; j < n; j += (long long)gridDim.x * blockDim.x)
        keys[j] = (unsigned long long)__double_as_longlong(load_logx(x, in_f32, base + j));
}
__global__ void k_pilot_pick(const unsigned long long *sorted, long long n, double *pilot)
{
    const double hi = __longlong_as_double((long long)sorted[n / 2]);
    *pilot = (n & 1) ? hi : (__longlong_as_double((long long)sorted[n / 2 - 1]) + hi) / 2.0;      // np.median: mean of the two middle values
}

int pilot_offsets(const void *d_x, int in_f32, long long rows, long long n, long long row_stride, double *d_pilot,
                  cudaStream_t st, int exact)
{
    if (!exact || n <= PILOT_CAP) {
        k_pilot<<<(unsigned)rows, 256, 0, st>>>(d_x, in_f32, n, row_stride, d_pilot);
        RB_LAUNCH_CHECK();
        return 0;
    }
    if (n > 0x7fffffffLL) return ST_INVALID;
    Arena ar(st);
    unsigned long long *k0 = nullptr, *k1 = nullptr;
    char *tmp = nullptr;
    size_t tmp_bytes = 0;
    RB_TRY(ar.alloc(&k0, (size_t)n));
    RB_TRY(ar.alloc(&k1, (size_t)n));
    cub::DeviceRadixSort::SortKeys(nullptr, tmp_bytes, k0, k1, (int)n, 0, 64, st);
    RB_TRY(ar.alloc(&tmp, tmp_bytes));
    const int blocks = (int)std::min<long long>((n + 255) / 256, 148 * 16);
    for (long long r = 0; r < rows; ++r) {
        k_pilot_keys<<<blocks, 256, 0, st>>>(d_x, in_f32, n, r * row_stride, k0);
        RB_LAUNCH_CHECK();
        RB_CUDA(cub::DeviceRadixSort::SortKeys(tmp, tmp_bytes, k0, k1, (int)n, 0, 64, st));
        count_launch(8);
        k_pilot_pick<<<1, 1, 0, st>>>(k1, n, d_pilot + r);
        RB_LAUNCH_CHECK();
    }
    return 0;
}

// ------------------------------------------------------------------ rolling AR(1) innovation variance
constexpr int RV_ITEMS = 8;

struct WinSums { double s1, s2, sl; };

__global__ void __launch_bounds__(256) k_rollvar(const double *__restrict__ C, long long n, long long row_stride, int w,
                                                 double *__restrict__ V)
{
    const long long row = blockIdx.y;
    const double *c = C + row * row_stride;
    double *v = V + row * row_stride;
    const long long j0 = ((long long)blockIdx.x * blockDim.x + threadIdx.x) * RV_ITEMS;
    if (j0 >= n) return;
    const long long half = w / 2, last = n - w;
    const double wd = (double)w, pairs = (double)(w - 1), rwd = 1.0 / wd, shrink = 1.0 + 1.0 / (wd + 1.0) + 1.0e-4;      // c1 of ar1_window_variance
    WinSums ws{0.0, 0.0, 0.0};
    long long tprev = -1;
    double cur = 0.0;
#pragma unroll 1
    for (int jj = 0; jj < RV_ITEMS; ++jj) {
        const long long j = j0 + jj;
        if (j >= n) break;
        long long t = j - half;
        if (t < 0) t = 0; else if (t > last) t = last;
        if (t != tprev) {
            if (tprev < 0) {
                ws.s1 = ws.s2 = ws.sl = 0.0;
                for (int k = 0; k < w; ++k) {
                    const double a = c[t + k];
                    ws.s1 = __dadd_rn(ws.s1, a);
                    ws.s2 = __fma_rn(a, a, ws.s2);
                    if (k < w - 1) ws.sl = __fma_rn(a, c[t + k + 1], ws.sl);
                }
            } else {
                // slide tprev -> t (= tprev + 1), wls_backend.c:714-724
                const double out_v = c[tprev], nx = c[tprev + w], lag_l = c[tprev + w - 1], lag_r = c[tprev + 1];
                ws.s1 = __dadd_rn(__dsub_rn(ws.s1, out_v), nx);
                ws.s2 = __fma_rn(nx, nx, __fma_rn(-out_v, out_v, ws.s2));
                ws.sl = __fma_rn(lag_l, nx, __fma_rn(-out_v, lag_r, ws.sl));
            }
            cur = ar1_window_variance(ws.s1, ws.s2, ws.sl, c[t], c[t + w - 1], wd, rwd, pairs, shrink);
            tprev = t;
        }
        v[j] = fmax(cur, 1.0e-8);                          // wls_backend.c:869
    }
}

// n < 5 (window 0) or n < 4: per-row robust scale^2 for both variance tracks (wls_backend.c:834-848)
__global__ void k_robust_rows(const double *C, long long n, long long row_stride, double *row_const)
{
    const long long row = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    if (row >= gridDim.x * (long long)blockDim.x) return;
    double buf[4];
    const int m = (int)n;                                  // n <= 4 here
    for (int k = 0; k < m; ++k) buf[k] = C[row * row_stride + k];
    auto med = [&](double *a, int len) {
        for (int i = 1; i < len; ++i) { double key = a[i]; int q = i; while (q > 0 && a[q - 1] > key) { a[q] = a[q - 1]; --q; } a[q] = key; }
        if (len == 1) return a[0];
        return (len & 1) ? a[len / 2] : 0.5 * (a[len / 2 - 1] + a[len / 2]);
    };
    const double m0 = med(buf, m);
    for (int k = 0; k < m; ++k) buf[k] = fabs(C[row * row_stride + k] - m0);
    double mad = med(buf, m);
    mad = __dmul_rn(mad, 1.4826);
    double sc = (mad > 1.0e-6) ? mad : 1.0e-6;
    row_const[row] = fmax(__dmul_rn(sc, sc), 1.0e-8);
}

// ------------------------------------------------------------------ trend knots from exact order statistics (sort-based)
constexpr unsigned long long YBASE = 0x3E10000000000000ULL;   // bits of 2^-30

__global__ void k_make_keys(const double *C, const double *V, long long n, unsigned long long *ky, unsigned long long *kx)
{
    for (long long j = (long long)blockIdx.x * blockDim.x + threadIdx.x; j < n; j += (long long)gridDim.x * blockDim.x) {
        ky[j] = (unsigned long long)__double_as_longlong(V[j]);           // V >= 1e-8 > 0: bit pattern is order preserving
        kx[j] = (unsigned long long)__double_as_longlong(fabs(C[j]));
    }
}

__device__ __forceinline__ int bin_of_rank(long long p, long long N, int B)
{
    int b = (int)((p * B) / N);
    if (b >= B) b = B - 1;
    while (b + 1 < B && ((long long)(b + 1) * N) / B <= p) ++b;
    while (b > 0 && ((long long)b * N) / B > p) --b;
    return b;
}

// after the lexicographic (x, y) sort: tag every y with its equal-count bin so one more sort groups y by bin
__global__ void k_bin_keys(const unsigned long long *ysorted, long long N, int B, unsigned long long *out)
{
    for (long long p = (long long)blockIdx.x * blockDim.x + threadIdx.x; p < N; p += (long long)gridDim.x * blockDim.x) {
        const unsigned long long yb = ysorted[p];
        unsigned long long rel = yb > YBASE ? yb - YBASE : 0ULL;
        if (rel >= (1ULL << 58)) rel = (1ULL << 58) - 1;
        out[p] = ((unsigned long long)bin_of_rank(p, N, B) << 58) | rel;
    }
}

// one thread per row: bin medians -> PAVA -> de-duplicated knots (wls_backend.c:476-560)
__global__ void k_knots_from_sorted(const unsigned long long *xsorted, const unsigned long long *ybinsorted, long long N, int B,
                                    Knots *out)
{
    if (threadIdx.x != 0 || blockIdx.x != 0) return;
    double bx[MAX_KNOTS], by[MAX_KNOTS], bw[MAX_KNOTS];
    int used = 0;
    for (int b = 0; b < B; ++b) {
        const long long lo = ((long long)b * N) / B, hi = ((long long)(b + 1) * N) / B;
        if (hi <= lo) continue;
        const long long wdt = hi - lo;
        auto xat = [&](long long p) { return __longlong_as_double((long long)xsorted[p]); };
        auto yat = [&](long long p) { return __longlong_as_double((long long)((ybinsorted[p] & ((1ULL << 58) - 1)) + YBASE)); };
        bx[used] = (wdt & 1) ? xat(lo + wdt / 2) : 0.5 * (xat(lo + wdt / 2 - 1) + xat(lo + wdt / 2));
        by[used] = (wdt & 1) ? yat(lo + wdt / 2) : 0.5 * (yat(lo + wdt / 2 - 1) + yat(lo + wdt / 2));
        if (wdt == 1) by[used] = yat(lo);
        bw[used] = (double)wdt;
        ++used;
    }
    knots_from_bins(bx, by, bw, used, out);
}

static int trend_knots_sorted(const double *d_C, const double *d_V, const std::vector<long long> &rows, long long n,
                              long long row_stride, Knots *d_knots, cudaStream_t st)
{
    const long long N = n;
    const int B = (int)fmax(4.0, floor(1.0 + (log((double)N + 1.0) / log(2.0))));      // wls_backend.c:456
    if (B > MAX_KNOTS) return ST_INVALID;
    Arena ar(st);
    unsigned long long *k0 = nullptr, *k1 = nullptr, *v0 = nullptr, *v1 = nullptr;
    RB_TRY(ar.alloc(&k0, (size_t)n)); RB_TRY(ar.alloc(&k1, (size_t)n));
    RB_TRY(ar.alloc(&v0, (size_t)n)); RB_TRY(ar.alloc(&v1, (size_t)n));
    size_t tmp_bytes = 0, tb2 = 0;
    cub::DeviceRadixSort::SortPairs(nullptr, tmp_bytes, k0, k1, v0, v1, (int)n, 0, 63, st);
    cub::DeviceRadixSort::SortKeys(nullptr, tb2, k0, k1, (int)n, 0, 64, st);
    tmp_bytes = std::max(tmp_bytes, tb2);
    char *tmp = nullptr;
    RB_TRY(ar.alloc(&tmp, tmp_bytes));
    const int blocks = (int)std::min<long long>((n + 255) / 256, 148 * 16);
    for (long long r : rows) {
        const double *c = d_C + r * row_stride, *v = d_V + r * row_stride;
        k_make_keys<<<blocks, 256, 0, st>>>(c, v, n, k0, v0);                 // k0 = y bits, v0 = x bits
        RB_LAUNCH_CHECK();
        RB_CUDA(cub::DeviceRadixSort::SortPairs(tmp, tmp_bytes, k0, k1, v0, v1, (int)n, 0, 63, st));   // by y
        count_launch(8);
        RB_CUDA(cub::DeviceRadixSort::SortPairs(tmp, tmp_bytes, v1, v0, k1, k0, (int)n, 0, 63, st));   // stable by x: v0 = x sorted, k0 = y
        count_launch(8);
        k_bin_keys<<<blocks, 256, 0, st>>>(k0, N, B, k1);
        RB_LAUNCH_CHECK();
        RB_CUDA(cub::DeviceRadixSort::SortKeys(tmp, tmp_bytes, k1, v1, (int)n, 0, 64, st));           // v1 = (bin, y) sorted
        count_launch(8);
        k_knots_from_sorted<<<1, 32, 0, st>>>(v0, v1, N, B, d_knots + r);
        RB_LAUNCH_CHECK();
    }
    return 0;
}

// 0: histogram multi-select with sort fallback (default); 1: force the sort-based path (tests)
static std::atomic<int> g_trend_mode{0};
static std::atomic<long long> g_trend_fallback_rows{0};
static std::atomic<long long> g_trend_fb_reason[8];

// ------------------------------------------------------------------ knot tables for the combine
// The trend of a row as the combine reads it: knots as {x, y} pairs, the slope of every segment, a 256-entry bucket -> first
// candidate segment table keyed by the exponent and the top four mantissa bits of |signal| (16 octaves from 2^-12), and the
// clamp range.  lin-interp with flat extrapolation (wls_backend.c:341-391) is then: clamp t to [x_0, x_last], start at
// lut[bucket(t)], step forward while the next knot is <= t (the knots are quantiles of |signal|, at most ~6 per octave:
// with 16 buckets per octave a warp rarely needs a step), y_lo + (t - x_lo) * slope_lo.
constexpr int KT_KNOTS = 32, KT_LUT = 256, KT_BASE = (1023 - 12) << 4;
struct KnotTable {
    double2 xy[KT_KNOTS];
    double slope[KT_KNOTS];
    unsigned char lut[KT_LUT];
    double xlo, xhi;
    int top;                      // last segment index (nk - 2, at least 0)
    int pad[3];
};
static_assert(sizeof(KnotTable) % 16 == 0, "KnotTable is staged with 128-bit copies");

__device__ __forceinline__ int knot_bucket(double t)
{
    const int key = (__double2hiint(t) >> 16) - KT_BASE;              // t >= 0: sign bit clear
    return min(max(key, 0), KT_LUT - 1);
}

__global__ void __launch_bounds__(KT_LUT) k_knot_tables(const Knots *knots, KnotTable *tables)
{
    const Knots &K = knots[blockIdx.x];
    KnotTable &T = tables[blockIdx.x];
    const int k = threadIdx.x;
    // a constant trend (one knot, or none) is a single flat segment at x = 0
    const bool flat = K.constant || K.nk <= 0;
    const int nk = flat ? 1 : K.nk;
    const double yflat = K.constant ? K.cval : 1.0e-8;
    if (k < KT_KNOTS) {
        const bool in = k < nk;
        T.xy[k] = make_double2(in ? (flat ? 0.0 : K.x[k]) : INFINITY, in ? (flat ? yflat : K.y[k]) : 0.0);
        double sl = 0.0;
        if (!flat && k + 1 < nk && K.x[k + 1] > K.x[k]) sl = (K.y[k + 1] - K.y[k]) / (K.x[k + 1] - K.x[k]);
        T.slope[k] = sl;
    }
    const int top = max(nk - 2, 0);
    if (k == 0) {
        T.top = top;
        T.xlo = flat ? 0.0 : K.x[0];
        T.xhi = flat ? 0.0 : K.x[nk - 1];
        T.pad[0] = T.pad[1] = T.pad[2] = 0;
    }
    // lut[b] = last segment whose left knot is <= the bucket's lower edge (bucket 0 also takes everything below it)
    const double edge = (k == 0) ? 0.0 : ldexp(1.0 + 0.0625 * (double)(k & 15), (k >> 4) - 12);
    int lo = 0;
    if (!flat)
        for (int q = 1; q <= top; ++q) if (K.x[q] <= edge) lo = q;
    T.lut[k] = (unsigned char)lo;
}

// ------------------------------------------------------------------ fused posterior + column reduction over samples
struct CombineParams {
    const double *C; const double *V; const KnotTable *tables; const double *row_const;
    long long m, n, row_stride;
    double ldf, pdf, tdf, pfr, lower_bound_z, min_effect;
    int use_min_effect; int const_rows;
    double *scores, *mean, *raw, *prior, *mod, *se;
    double *acc;          // != nullptr: sample-sharded mode, write the per-bin sums [4][n] ([2][n] without WANT_RQ) and stop
    int *bad;
};

constexpr int CB_THREADS = 512;           // two CTAs per SM: one stages its tables while the other computes
constexpr int CB_ROWS_SMEM = 40;          // knot tables staged per batch of sample rows (41 KB)

// posterior precision of one sample-bin and its accumulation (wls_backend.c:889-911)
template <bool WANT_RQ>
__device__ __forceinline__ void combine_one(double y, double ov, double pv, double ldf, double pdf, double rtdf1, double pfr,
                                            double &wsum, double &psum, double &rsum, double &qsum)
{
    double post = __fma_rn(ldf, ov, pdf * pv) * rtdf1;
    post = dmax(dmax(post, pfr * pv), 1.0e-8);
    const double prec = rcp_nr(post);                 // 1 / post to ~1 ulp (hardware seed + two Newton steps)
    if (WANT_RQ) { rsum += rcp_nr(ov); qsum += rcp_nr(pv); }
    psum += prec;
    wsum = __fma_rn(prec, y, wsum);
}

template <bool CONST_ROWS, bool WANT_RQ>
__global__ void __launch_bounds__(CB_THREADS, 2) k_combine(CombineParams P)
{
    __shared__ __align__(16) KnotTable s_t[CONST_ROWS ? 1 : CB_ROWS_SMEM];
    const long long j = (long long)blockIdx.x * CB_THREADS + threadIdx.x;
    const bool live = j < P.n;
    double wsum = 0.0, psum = 0.0, rsum = 0.0, qsum = 0.0;
    const double rtdf1 = 1.0 / fmax(P.tdf, 1.0);
    const double ldf = P.ldf, pdf = P.pdf, pfr = P.pfr;
    const long long stride = P.row_stride;
    if (CONST_ROWS) {
        if (live) {
            const double *pc = P.C + j;
            for (long long r = 0; r < P.m; ++r, pc += stride) {
                const double v = P.row_const[r];
                combine_one<WANT_RQ>(*pc, v, v, ldf, pdf, rtdf1, pfr, wsum, psum, rsum, qsum);
            }
        }
    } else {
        const double *pc = P.C + (live ? j : 0), *pv_ = P.V + (live ? j : 0);
        for (long long r0 = 0; r0 < P.m; r0 += CB_ROWS_SMEM) {
            const int nr = (int)min((long long)CB_ROWS_SMEM, P.m - r0);
            __syncthreads();
            {
                const uint4 *src = reinterpret_cast<const uint4 *>(P.tables + r0);
                uint4 *dst = reinterpret_cast<uint4 *>(s_t);
                for (int e = threadIdx.x; e < nr * (int)(sizeof(KnotTable) / 16); e += CB_THREADS) dst[e] = src[e];
            }
            __syncthreads();
            if (live) {
                // rows in groups of four: the eight loads of a group are issued before any of its arithmetic
                for (int rb = 0; rb < nr; rb += 4) {
                    double ys[4], vs[4];
#pragma unroll
                    for (int u = 0; u < 4; ++u) {
                        const bool in = rb + u < nr;
                        ys[u] = in ? pc[(long long)u * stride] : 0.0;
                        vs[u] = in ? pv_[(long long)u * stride] : 1.0;
                    }
#pragma unroll
                    for (int u = 0; u < 4; ++u) {
                        if (rb + u >= nr) break;
                        const KnotTable &T = s_t[rb + u];
                        const double tt = dmin(dmax(fabs(ys[u]), T.xlo), T.xhi);
                        int lo = T.lut[knot_bucket(tt)];
                        const int top = T.top;
                        while (lo < top && T.xy[lo + 1].x <= tt) ++lo;
                        const double2 k = T.xy[lo];
                        const double pv = dmax(__fma_rn(tt - k.x, T.slope[lo], k.y), 1.0e-8);
                        combine_one<WANT_RQ>(ys[u], vs[u], pv, ldf, pdf, rtdf1, pfr, wsum, psum, rsum, qsum);     // V is floored at 1e-8 by its producer
                    }
                    const int adv = min(4, nr - rb);
                    pc += (long long)adv * stride; pv_ += (long long)adv * stride;
                }
            }
        }
    }
    if (!live) return;
    if (P.acc) {                                   // partial sums of this rank's samples (summed across ranks by the caller)
        P.acc[j] = wsum; P.acc[P.n + j] = psum;
        if (WANT_RQ) { P.acc[2 * P.n + j] = rsum; P.acc[3 * P.n + j] = qsum; }
        return;
    }
    // wls_backend.c:915-937
    const double Pj = fmax(psum, 1.0e-8);
    const double mean = wsum / Pj;
    const double md = (double)P.m;
    const double se = sqrt(1.0 / Pj);
    const double z = mean / fmax(se, 1.0e-8);
    const double sc = P.use_min_effect ? __dsub_rn(mean, fmax(P.min_effect, 0.0)) / fmax(se, 1.0e-8) : __dsub_rn(z, P.lower_bound_z);
    const double rawv = md / fmax(rsum, 1.0e-8), priv = md / fmax(qsum, 1.0e-8), modv = md / Pj;
    if (!(isfinite(sc) && isfinite(mean) && isfinite(rawv) && isfinite(priv) && isfinite(modv) && isfinite(se) && isfinite(z)))
        *P.bad = 1;
    if (P.scores) P.scores[j] = sc;
    if (P.mean) P.mean[j] = mean;
    if (P.raw) P.raw[j] = rawv;
    if (P.prior) P.prior[j] = priv;
    if (P.mod) P.mod[j] = modv;
    if (P.se) P.se[j] = se;
}

// finalisation of summed accumulators (sample-sharded scoring): wls_backend.c:915-937 on [4][n] sums, or on [2][n] when
// only the scores and the mean are wanted (has_rq = 0: the raw / prior variance rows are absent)
__global__ void __launch_bounds__(256) k_finalize_acc(const double *acc, long long n, int has_rq, double m_total, double lower_bound_z,
                                                      double min_effect, int use_min_effect, double *scores, double *mean_o,
                                                      double *raw, double *prior, double *mod, double *se_o, int *bad)
{
    const long long j = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= n) return;
    const double wsum = acc[j], psum = acc[n + j];
    const double rsum = has_rq ? acc[2 * n + j] : 1.0, qsum = has_rq ? acc[3 * n + j] : 1.0;
    const double Pj = fmax(psum, 1.0e-8);
    const double mean = wsum / Pj;
    const double se = sqrt(1.0 / Pj);
    const double z = mean / fmax(se, 1.0e-8);
    const double sc = use_min_effect ? __dsub_rn(mean, fmax(min_effect, 0.0)) / fmax(se, 1.0e-8) : __dsub_rn(z, lower_bound_z);
    const double rawv = m_total / fmax(rsum, 1.0e-8), priv = m_total / fmax(qsum, 1.0e-8), modv = m_total / Pj;
    if (!(isfinite(sc) && isfinite(mean) && isfinite(rawv) && isfinite(priv) && isfinite(modv) && isfinite(se))) *bad = 1;
    if (scores) scores[j] = sc;
    if (mean_o) mean_o[j] = mean;
    if (raw) raw[j] = rawv;
    if (prior) prior[j] = priv;
    if (mod) mod[j] = modv;
    if (se_o) se_o[j] = se;
}

// ---- the per-row stages (rolling variance + trend knots) and the cross-sample finish, split so that the host
// ---- entry can pipeline row groups behind their host->device copies
struct WlsRun {
    long long m = 0, n = 0;
    int w = 0;
    double ldf = 0, pdf = 0, tdf = 0, pfr = 0;
    bool const_rows = false, fused = false, sort_all = false;
    double *d_V = nullptr, *d_rc = nullptr;
    Knots *d_knots = nullptr;
    KnotTable *d_tables = nullptr;
    int *d_fb = nullptr, *d_bad = nullptr;
};

static int wls_prepare(Arena &ar, long long m, long long n, const rocco_b200_score_params &prm, rocco_b200_score_outputs *out,
                       WlsRun &R, cudaStream_t st)
{
    R.m = m; R.n = n;
    R.pdf = fmax(prm.prior_df, 0.0); R.pfr = fmax(prm.precision_floor_ratio, 0.0);
    R.w = resolve_spatial_window(n, prm.spatial_window);
    R.ldf = R.w > 0 ? fmax(4.0, (double)R.w - 3.0) : 1.0;
    R.tdf = R.ldf + R.pdf;
    out->total_df = R.tdf;
    out->resolved_spatial_window = R.w;
    RB_TRY(ar.alloc(&R.d_bad, 1));
    RB_CUDA(cudaMemsetAsync(R.d_bad, 0, sizeof(int), st));
    R.const_rows = (R.w == 0 || n < 4);
    if (R.const_rows) {
        RB_TRY(ar.alloc(&R.d_rc, (size_t)m));
    } else {
        RB_TRY(ar.alloc(&R.d_V, (size_t)m * n));
        RB_TRY(ar.alloc(&R.d_knots, (size_t)m));
        RB_TRY(ar.alloc(&R.d_tables, (size_t)m));
        RB_TRY(ar.alloc(&R.d_fb, (size_t)m));
        R.sort_all = g_trend_mode.load() == 1;
        R.fused = !R.sort_all && (R.w <= trend_fused_max_window());
    }
    return 0;
}

// rows [r0, r1): variance track and trend knots (everything that needs one sample row only)
static int wls_rows(const double *d_centered, WlsRun &R, long long r0, long long r1, cudaStream_t st)
{
    const long long g = r1 - r0, n = R.n;
    const double *c = d_centered + r0 * n;
    if (R.const_rows) {
        k_robust_rows<<<(unsigned)g, 1, 0, st>>>(c, n, n, R.d_rc + r0);
        RB_LAUNCH_CHECK();
        return 0;
    }
    double *v = R.d_V + r0 * n;
    if (!R.fused) {
        dim3 grid((unsigned)((n + 256LL * RV_ITEMS - 1) / (256LL * RV_ITEMS)), (unsigned)g);
        RB_PROF("k_rollvar", st, (double)g * (double)n * 16.0);
        k_rollvar<<<grid, 256, 0, st>>>(c, n, n, R.w, v);
        RB_LAUNCH_CHECK();
    }
    if (!R.sort_all) RB_TRY(trend_knots_select(c, v, g, n, n, R.d_knots + r0, R.d_fb + r0, R.fused ? R.w : 0, st));
    return 0;
}

// after every row went through wls_rows: sort-path for flagged rows, then the fused column reduction
// d_acc != nullptr: write the per-bin sums instead of the outputs -- all four rows with acc_rq, else {sum y/post, sum 1/post}
static int wls_finish(const double *d_centered, WlsRun &R, const rocco_b200_score_params &prm, rocco_b200_score_outputs *out,
                      cudaStream_t st, double *d_acc = nullptr, bool acc_rq = true)
{
    const long long m = R.m, n = R.n;
    CombineParams P{};
    P.C = d_centered; P.m = m; P.n = n; P.row_stride = n;
    P.ldf = R.ldf; P.pdf = R.pdf; P.tdf = R.tdf; P.pfr = R.pfr; P.lower_bound_z = prm.lower_bound_z;
    P.min_effect = prm.min_effect; P.use_min_effect = prm.use_min_effect;
    P.scores = out->scores; P.mean = out->mean; P.raw = out->raw_variance; P.prior = out->prior_variance;
    P.mod = out->moderated_variance; P.se = out->standard_error; P.bad = R.d_bad; P.acc = d_acc;
    if (R.const_rows) {
        P.const_rows = 1; P.row_const = R.d_rc;
    } else {
        // exact order statistics by histogram multi-select; rows it flags (a bucket over capacity: massive ties)
        // fall back to the sort-based path, which is exact for any input
        std::vector<long long> rows;
        if (R.sort_all) {
            for (long long r = 0; r < m; ++r) rows.push_back(r);
        } else {
            std::vector<int> fb((size_t)m);
            RB_CUDA(cudaMemcpyAsync(fb.data(), R.d_fb, sizeof(int) * (size_t)m, cudaMemcpyDeviceToHost, st));
            RB_CUDA(cudaStreamSynchronize(st));
            for (long long r = 0; r < m; ++r)
                if (fb[(size_t)r]) { rows.push_back(r); for (int k = 0; k < 8; ++k) if (fb[(size_t)r] & (1 << k)) g_trend_fb_reason[k].fetch_add(1); }
        }
        if (!rows.empty()) {
            g_trend_fallback_rows.fetch_add((long long)rows.size());
            RB_PROF("trend_sort_fallback", st, (double)rows.size() * (double)n * 16.0);
            RB_TRY(trend_knots_sorted(d_centered, R.d_V, rows, n, n, R.d_knots, st));
        }
        P.const_rows = 0; P.V = R.d_V; P.tables = R.d_tables;
        k_knot_tables<<<(unsigned)m, KT_LUT, 0, st>>>(R.d_knots, R.d_tables);
        RB_LAUNCH_CHECK();
    }
    {
        RB_PROF("k_combine", st, (double)m * (double)n * (P.const_rows ? 8.0 : 16.0) + 48.0 * (double)n);
        const unsigned grid = (unsigned)((n + CB_THREADS - 1) / CB_THREADS);
        const bool want_rq = P.acc ? acc_rq : (P.raw != nullptr) || (P.prior != nullptr);   // raw / prior variance sums only when asked for
        if (P.const_rows) {
            if (want_rq) k_combine<true, true><<<grid, CB_THREADS, 0, st>>>(P); else k_combine<true, false><<<grid, CB_THREADS, 0, st>>>(P);
        } else {
            if (want_rq) k_combine<false, true><<<grid, CB_THREADS, 0, st>>>(P); else k_combine<false, false><<<grid, CB_THREADS, 0, st>>>(P);
        }
        RB_LAUNCH_CHECK();
    }
    int bad = 0;
    RB_CUDA(cudaMemcpyAsync(&bad, R.d_bad, sizeof(int), cudaMemcpyDeviceToHost, st));
    RB_CUDA(cudaStreamSynchronize(st));
    if (bad) return ST_NONFINITE;
    return 0;
}

int centered_wls(const double *d_centered, long long m, long long n, const rocco_b200_score_params &prm,
                 rocco_b200_score_outputs *out, cudaStream_t st, double *d_acc2)
{
    if (!d_centered || !out || m <= 0 || n <= 0) return ST_INVALID;
    Arena ar(st);
    WlsRun R;
    RB_TRY(wls_prepare(ar, m, n, prm, out, R, st));
    RB_TRY(wls_rows(d_centered, R, 0, m, st));
    return wls_finish(d_centered, R, prm, out, st, d_acc2, false);
}

int finalize_acc(const double *d_acc, long long n, bool has_rq, long long m_total, const rocco_b200_score_params &prm,
                 rocco_b200_score_outputs *out, int *d_bad, cudaStream_t st)
{
    k_finalize_acc<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(d_acc, n, has_rq ? 1 : 0, (double)m_total, prm.lower_bound_z,
                                                                prm.min_effect, prm.use_min_effect, out->scores, out->mean,
                                                                out->raw_variance, out->prior_variance, out->moderated_variance,
                                                                out->standard_error, d_bad);
    RB_LAUNCH_CHECK();
    return 0;
}

// ------------------------------------------------------------------ the full chain (inference.py:302-379)
// `h_matrix` != nullptr: the matrix lives on the host; row groups are copied on a second stream and every
// per-row stage of a group starts as soon as its rows have landed (copy of group g+1 overlaps compute of g).
static cudaStream_t copy_stream()
{
    static cudaStream_t cs[32] = {nullptr};
    static std::mutex mu;                      // first use races between host threads otherwise (a half-created handle is visible)
    int dev = 0;
    cudaGetDevice(&dev);
    dev &= 31;
    std::lock_guard<std::mutex> lk(mu);
    if (!cs[dev]) {
        cudaStream_t s = nullptr;
        if (cudaStreamCreateWithFlags(&s, cudaStreamNonBlocking) != cudaSuccess) { (void)cudaGetLastError(); s = nullptr; }
        cs[dev] = s;
    }
    return cs[dev];
}

// Pageable caller memory (what a NumPy array is): a cudaMemcpyAsync from it is staged by the driver through its own
// small pinned buffer by ONE thread at a fraction of the link rate, and blocks the caller meanwhile.  The matrix is
// instead copied into a ring of pinned chunks by several host threads (the copy is memory-bandwidth bound: one core
// moves ~10 GB/s, the link takes 55) and each chunk goes to the device as a true asynchronous DMA while the next one
// is being filled.  (cudaHostRegister on the caller's buffer would avoid the extra pass but costs ~0.2 s per GB of
// page pinning, more than the copy itself.)
class StageCopier {
  public:
    static StageCopier &get() { static StageCopier *inst = new StageCopier(); return *inst; }     // never destroyed: worker threads outlive main
    void copy(char *dst, const char *src, size_t bytes)
    {
        const size_t piece = std::max<size_t>((size_t)1 << 20, (bytes + nthreads_) / (nthreads_ + 1));
        {
            std::lock_guard<std::mutex> lk(mu_);
            for (size_t off = 0; off < bytes; off += piece) { jobs_.push_back({dst + off, src + off, std::min(piece, bytes - off)}); ++pending_; }
        }
        cv_.notify_all();
        for (;;) {                                    // the caller works too
            Job j;
            {
                std::lock_guard<std::mutex> lk(mu_);
                if (jobs_.empty()) break;
                j = jobs_.front(); jobs_.pop_front();
            }
            memcpy(j.dst, j.src, j.n);
            finish_one();
        }
        std::unique_lock<std::mutex> lk(mu_);
        done_.wait(lk, [&] { return pending_ == 0; });
    }

  private:
    struct Job { char *dst; const char *src; size_t n; };
    StageCopier()
    {
        // the copy is bound by what one core can move (4-10 GB/s), so it takes most of the cores this process may claim: all
        // but one of the host's, divided by the ranks that share the host (torchrun's LOCAL_WORLD_SIZE), at most 15 helpers
        unsigned hw = std::thread::hardware_concurrency();
        unsigned ranks = 1;
        if (const char *e = getenv("ROCCO_B200_STAGE_THREADS")) { nthreads_ = std::max(0, std::min(63, atoi(e))); ranks = 0; }
        else if (const char *e = getenv("LOCAL_WORLD_SIZE")) ranks = (unsigned)std::max(1, atoi(e));
        if (ranks) nthreads_ = (int)std::max(1u, std::min(15u, (hw ? hw : 2u) / ranks > 1 ? (hw ? hw : 2u) / ranks - 1 : 1u));
        for (int t = 0; t < nthreads_; ++t) std::thread([this] { worker(); }).detach();
    }
    void finish_one()
    {
        std::lock_guard<std::mutex> lk(mu_);
        if (--pending_ == 0) done_.notify_all();
    }
    void worker()
    {
        for (;;) {
            Job j;
            {
                std::unique_lock<std::mutex> lk(mu_);
                cv_.wait(lk, [&] { return !jobs_.empty(); });
                j = jobs_.front(); jobs_.pop_front();
            }
            memcpy(j.dst, j.src, j.n);
            finish_one();
        }
    }
    std::mutex mu_;
    std::condition_variable cv_, done_;
    std::deque<Job> jobs_;
    int pending_ = 0;
    int nthreads_ = 1;
};

constexpr int STAGE_SLOTS = 4;
constexpr size_t STAGE_CHUNK = (size_t)32 << 20;
struct StageRing {
    char *buf[STAGE_SLOTS] = {nullptr, nullptr, nullptr, nullptr};
    cudaEvent_t done[STAGE_SLOTS] = {nullptr, nullptr, nullptr, nullptr};
    bool used[STAGE_SLOTS] = {false, false, false, false};
    int next = 0;
    bool ok = false;
};
// one ring per device, created on first use; only touched under the copy mutex of score_loci_core
static StageRing *stage_ring()
{
    static StageRing rings[32];
    int dev = 0;
    cudaGetDevice(&dev);
    StageRing &R = rings[dev & 31];
    if (!R.ok) {
        bool good = true;
        for (int k = 0; k < STAGE_SLOTS && good; ++k) {
            good = cudaMallocHost(reinterpret_cast<void **>(&R.buf[k]), STAGE_CHUNK) == cudaSuccess &&
                   cudaEventCreateWithFlags(&R.done[k], cudaEventDisableTiming) == cudaSuccess;
        }
        if (!good) { (void)cudaGetLastError(); return nullptr; }
        R.ok = true;
    }
    return &R;
}

static bool host_pointer_is_pinned(const void *p)
{
    cudaPointerAttributes at{};
    if (cudaPointerGetAttributes(&at, p) != cudaSuccess) { (void)cudaGetLastError(); return false; }
    return at.type == cudaMemoryTypeHost || at.type == cudaMemoryTypeManaged;
}

// host -> device copy of `bytes` on stream cs: direct DMA for pinned memory, the staged ring otherwise
static int upload_rows(char *d_dst, const char *h_src, size_t bytes, bool pinned, cudaStream_t cs)
{
    StageRing *R = pinned ? nullptr : stage_ring();
    if (!R) {
        RB_CUDA(cudaMemcpyAsync(d_dst, h_src, bytes, cudaMemcpyHostToDevice, cs));
        return 0;
    }
    for (size_t off = 0; off < bytes; off += STAGE_CHUNK) {
        const size_t len = std::min(STAGE_CHUNK, bytes - off);
        const int k = R->next;
        R->next = (k + 1) % STAGE_SLOTS;
        if (R->used[k]) RB_CUDA(cudaEventSynchronize(R->done[k]));          // the DMA that last read this slot has finished
        StageCopier::get().copy(R->buf[k], h_src + off, len);
        RB_CUDA(cudaMemcpyAsync(d_dst + off, R->buf[k], len, cudaMemcpyHostToDevice, cs));
        RB_CUDA(cudaEventRecord(R->done[k], cs));
        R->used[k] = true;
    }
    return 0;
}

static int score_loci_core(const void *d_matrix_in, const void *h_matrix, int dtype, long long m, long long n,
                           const rocco_b200_score_params *params, rocco_b200_score_outputs *out, cudaStream_t st,
                           double *d_acc = nullptr)
{
    if ((!d_matrix_in && !h_matrix) || !out || m <= 0 || n <= 0 || (dtype != 0 && dtype != 1)) return ST_INVALID;
    rocco_b200_score_params prm;
    if (params) prm = *params; else rocco_b200_default_score_params(&prm);
    RB_TRY(ensure_device());
    Arena ar(st);
    const size_t esz = dtype ? sizeof(float) : sizeof(double);
    double *d_pilot = nullptr, *d_cent = nullptr;
    int *d_bad = nullptr;
    char *d_x = nullptr;
    RB_TRY(ar.alloc(&d_pilot, (size_t)m));
    RB_TRY(ar.alloc(&d_bad, 1));
    RB_CUDA(cudaMemsetAsync(d_bad, 0, sizeof(int), st));
    if (out->centered_matrix == nullptr) RB_TRY(ar.alloc(&d_cent, (size_t)m * n)); else d_cent = out->centered_matrix;
    const void *d_matrix = d_matrix_in;
    // row groups of ~256 MB
    long long group = std::max<long long>(1, std::min<long long>(m, (256LL << 20) / std::max<long long>(1, n * (long long)esz)));
    if (!h_matrix) group = m;
    const int ngroups = (int)((m + group - 1) / group);
    struct EventList {                            // destroyed on every exit path, including the early error returns
        std::vector<cudaEvent_t> v;
        ~EventList() { for (cudaEvent_t e : v) if (e) cudaEventDestroy(e); }
        cudaEvent_t &operator[](int i) { return v[(size_t)i]; }
    } ev;
    bool copies_queued = false;
    struct CopyDrain {                            // any exit after the uploads were queued waits for them before d_x is released
        const bool &on; cudaStream_t cs;
        ~CopyDrain() { if (on && cs) cudaStreamSynchronize(cs); }
    };
    cudaStream_t cs_drain = h_matrix ? copy_stream() : nullptr;
    CopyDrain drain{copies_queued, cs_drain};     // declared after the arena: runs before the arena frees d_x
    const int bw = resolve_baseline_window(n, prm.baseline_window > 0 ? prm.baseline_window : 101);
    const double lam = bw > 0 ? whittaker_lambda(bw) : 0.0;
    out->baseline_window = bw;
    out->baseline_lambda = lam;
    WlsRun R;
    RB_TRY(wls_prepare(ar, m, n, prm, out, R, st));
    // one call's row groups go into the shared copy stream back to back: concurrent callers then finish one after
    // the other at full PCIe rate (and start their next chromosome staggered) instead of all at once at 1/T of it
    static std::mutex copy_mu;
    std::unique_lock<std::mutex> copy_lock(copy_mu, std::defer_lock);
    bool pinned = true;
    cudaStream_t cs = cs_drain;
    if (h_matrix) {
        RB_TRY(ar.alloc(&d_x, (size_t)m * n * esz));
        d_matrix = d_x;
        copy_lock.lock();
        cudaEvent_t ready;
        RB_CUDA(cudaEventCreateWithFlags(&ready, cudaEventDisableTiming));
        RB_CUDA(cudaEventRecord(ready, st));                       // the stream-ordered allocation is valid from here on
        RB_CUDA(cudaStreamWaitEvent(cs, ready, 0));
        cudaEventDestroy(ready);
        ev.v.assign((size_t)ngroups, nullptr);
        pinned = host_pointer_is_pinned(h_matrix);
    }
    int status = 0;
    for (int g = 0; g < ngroups && status == 0; ++g) {
        const long long r0 = g * group, r1 = std::min(m, r0 + group);
        if (h_matrix) {
            // queue (pinned source) or stage-and-queue (pageable source) this group's rows, then launch its per-row stages
            // behind the copy: the kernels of group g run while the host stages group g+1
            copies_queued = true;
            status = upload_rows(d_x + (size_t)r0 * n * esz, (const char *)h_matrix + (size_t)r0 * n * esz,
                                 (size_t)(r1 - r0) * n * esz, pinned, cs);
            if (status != 0) break;
            RB_CUDA(cudaEventCreateWithFlags(&ev[g], cudaEventDisableTiming));
            RB_CUDA(cudaEventRecord(ev[g], cs));
            RB_CUDA(cudaStreamWaitEvent(st, ev[g], 0));
            if (g == ngroups - 1) copy_lock.unlock();
        }
        const char *xg = (const char *)d_matrix + (size_t)r0 * n * esz;
        {
            RB_PROF("k_pilot", st, 0.0);
            status = pilot_offsets(xg, dtype, r1 - r0, n, n, d_pilot + r0, st, prm.pilot_mode);
        }
        if (status == 0) status = whittaker_rows(xg, dtype, 1, d_pilot + r0, r1 - r0, n, n, lam, 0, d_cent + r0 * n, d_bad, st);
        if (status == 0) status = wls_rows(d_cent, R, r0, r1, st);
    }
    if (copy_lock.owns_lock()) copy_lock.unlock();
    if (status != 0) { cudaStreamSynchronize(st); return status; }
    int bad = 0;
    RB_CUDA(cudaMemcpyAsync(&bad, d_bad, sizeof(int), cudaMemcpyDeviceToHost, st));
    RB_CUDA(cudaStreamSynchronize(st));
    copies_queued = false;                        // st waited on every group's copy: nothing of this call is left in the copy stream
    if (bad) return ST_NONFINITE;
    return wls_finish(d_cent, R, prm, out, st, d_acc);
}

static int score_loci_dev(const void *d_matrix, int dtype, long long m, long long n, const rocco_b200_score_params *params,
                          rocco_b200_score_outputs *out, cudaStream_t st)
{
    return score_loci_core(d_matrix, nullptr, dtype, m, n, params, out, st);
}

}  // namespace score
}  // namespace rb

// ====================================================================== C-ABI
using namespace rb;
#define RB_API extern "C" __attribute__((visibility("default")))

RB_API int rocco_b200_trend_set_mode(int mode)
{
    return score::g_trend_mode.exchange(mode == 1 ? 1 : 0);
}
RB_API long long rocco_b200_trend_fallback_rows(void) { return score::g_trend_fallback_rows.load(); }
RB_API long long rocco_b200_whittaker_exact_rows(void) { return score::whittaker_exact_rows(); }
RB_API void rocco_b200_trend_fallback_reasons(long long *out8) { for (int k = 0; k < 8; ++k) out8[k] = score::g_trend_fb_reason[k].load(); }

RB_API void rocco_b200_default_score_params(rocco_b200_score_params *p)
{
    if (!p) return;
    p->lower_bound_z = 1.0; p->prior_df = 5.0; p->min_effect = 0.0; p->use_min_effect = 0;
    p->spatial_window = 31; p->precision_floor_ratio = 0.01; p->baseline_window = 101; p->pilot_mode = 0;
}

RB_API int rocco_b200_score_loci_wls_dev(const void *d_matrix, int dtype, size_t m, size_t n,
                                         const rocco_b200_score_params *params, rocco_b200_score_outputs *out, void *cuda_stream)
{
    return score::score_loci_dev(d_matrix, dtype, (long long)m, (long long)n, params, out, (cudaStream_t)cuda_stream);
}

/* Sample-sharded scoring: this rank's rows -> four per-bin sums [4][n]; sum them over ranks, then finalise.  The _ex form
 * also leaves the rank's centred rows in d_centered_out [m_local][n] (NULL: not kept). */
RB_API int rocco_b200_score_partial_ex_dev(const void *d_matrix, int dtype, size_t m_local, size_t n,
                                           const rocco_b200_score_params *params, double *d_centered_out, double *d_acc,
                                           void *cuda_stream)
{
    if (!d_acc) return ST_INVALID;
    rocco_b200_score_outputs out{};
    out.centered_matrix = d_centered_out;
    return score::score_loci_core(d_matrix, nullptr, dtype, (long long)m_local, (long long)n, params, &out, (cudaStream_t)cuda_stream, d_acc);
}

RB_API int rocco_b200_score_partial_dev(const void *d_matrix, int dtype, size_t m_local, size_t n,
                                        const rocco_b200_score_params *params, double *d_acc, void *cuda_stream)
{
    return rocco_b200_score_partial_ex_dev(d_matrix, dtype, m_local, n, params, nullptr, d_acc, cuda_stream);
}

RB_API int rocco_b200_score_finalize_dev(const double *d_acc, size_t m_total, size_t n, const rocco_b200_score_params *params,
                                         rocco_b200_score_outputs *out, void *cuda_stream)
{
    if (!d_acc || !out || m_total == 0 || n == 0) return ST_INVALID;
    rocco_b200_score_params prm;
    if (params) prm = *params; else rocco_b200_default_score_params(&prm);
    RB_TRY(ensure_device());
    cudaStream_t st = (cudaStream_t)cuda_stream;
    Arena ar(st);
    int *d_bad = nullptr;
    RB_TRY(ar.alloc(&d_bad, 1));
    RB_CUDA(cudaMemsetAsync(d_bad, 0, sizeof(int), st));
    RB_TRY(score::finalize_acc(d_acc, (long long)n, true, (long long)m_total, prm, out, d_bad, st));
    const int w = score::resolve_spatial_window((long long)n, prm.spatial_window);
    out->resolved_spatial_window = w;
    out->total_df = (w > 0 ? fmax(4.0, (double)w - 3.0) : 1.0) + fmax(prm.prior_df, 0.0);
    int bad = 0;
    RB_CUDA(cudaMemcpyAsync(&bad, d_bad, sizeof(int), cudaMemcpyDeviceToHost, st));
    RB_CUDA(cudaStreamSynchronize(st));
    return bad ? ST_NONFINITE : 0;
}

RB_API int rocco_b200_crossfit_baseline_dev(const double *d_rows, size_t m, size_t n, double penalty_lambda,
                                            double *d_out, void *cuda_stream)
{
    if (!d_rows || !d_out) return ST_NOMEM;                  // baseline_backend.c:313-316 returns -1 on NULL
    if (m == 0 || n == 0) return 0;
    RB_TRY(ensure_device());
    cudaStream_t st = (cudaStream_t)cuda_stream;
    Arena ar(st);
    int *d_bad = nullptr;
    RB_TRY(ar.alloc(&d_bad, 1));
    RB_CUDA(cudaMemsetAsync(d_bad, 0, sizeof(int), st));
    RB_TRY(score::whittaker_rows(d_rows, 0, 0, nullptr, (long long)m, (long long)n, (long long)n, penalty_lambda, 1, d_out, d_bad, st));
    RB_CUDA(cudaStreamSynchronize(st));
    return 0;
}

RB_API int rocco_b200_score_centered_wls_dev(const double *d_centered, size_t m, size_t n,
                                             const rocco_b200_score_params *params, rocco_b200_score_outputs *out,
                                             void *cuda_stream)
{
    if (!d_centered || !out || m == 0 || n == 0) return ST_INVALID;
    rocco_b200_score_params prm;
    if (params) prm = *params; else rocco_b200_default_score_params(&prm);
    RB_TRY(ensure_device());
    return score::centered_wls(d_centered, (long long)m, (long long)n, prm, out, (cudaStream_t)cuda_stream);
}

// ---- host-pointer entries (H2D / D2H inside)
namespace {
struct HostOuts {
    double *dev[6] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};
    double *host[6];
};
}

static int run_host_outputs(Arena &ar, size_t n, rocco_b200_score_outputs &host_out, rocco_b200_score_outputs &dev_out, HostOuts &ho)
{
    double **hp[6] = {&host_out.scores, &host_out.mean, &host_out.raw_variance, &host_out.prior_variance,
                      &host_out.moderated_variance, &host_out.standard_error};
    double **dp[6] = {&dev_out.scores, &dev_out.mean, &dev_out.raw_variance, &dev_out.prior_variance,
                      &dev_out.moderated_variance, &dev_out.standard_error};
    for (int k = 0; k < 6; ++k) {
        ho.host[k] = *hp[k];
        *dp[k] = nullptr;
        if (*hp[k]) { RB_TRY(ar.alloc(&ho.dev[k], n)); *dp[k] = ho.dev[k]; }
    }
    return 0;
}

static int copy_back(size_t n, HostOuts &ho, cudaStream_t st)
{
    for (int k = 0; k < 6; ++k)
        if (ho.host[k]) RB_CUDA(cudaMemcpyAsync(ho.host[k], ho.dev[k], n * sizeof(double), cudaMemcpyDeviceToHost, st));
    RB_CUDA(cudaStreamSynchronize(st));
    return 0;
}

static int score_loci_host(const void *matrix, int dtype, size_t m, size_t n, const rocco_b200_score_params *params,
                           rocco_b200_score_outputs *out)
{
    if (!matrix || !out || m == 0 || n == 0) return ST_INVALID;
    RB_TRY(ensure_device());
    // scratch of one call: input copy, centred matrix, variance track (m x n each) + ~1.5 GB of select / per-bin buffers
    HostScope lease(false, m * n * ((dtype ? sizeof(float) : sizeof(double)) + 16) + ((size_t)3 << 29));
    cudaStream_t st = lease.stream();
    Arena ar(st);
    rocco_b200_score_outputs dev = *out;
    HostOuts ho;
    RB_TRY(run_host_outputs(ar, n, *out, dev, ho));
    double *d_cent = nullptr;
    if (out->centered_matrix) { RB_TRY(ar.alloc(&d_cent, m * n)); }
    dev.centered_matrix = d_cent;
    int s = score::score_loci_core(nullptr, matrix, dtype, (long long)m, (long long)n, params, &dev, st);
    if (s != 0) return s;
    out->total_df = dev.total_df; out->resolved_spatial_window = dev.resolved_spatial_window;
    out->baseline_window = dev.baseline_window; out->baseline_lambda = dev.baseline_lambda;
    if (out->centered_matrix)
        RB_CUDA(cudaMemcpyAsync(out->centered_matrix, d_cent, m * n * sizeof(double), cudaMemcpyDeviceToHost, st));
    return copy_back(n, ho, st);
}

RB_API int rocco_score_loci_wls_f64(const double *matrix, size_t m, size_t n, const rocco_b200_score_params *params,
                                    rocco_b200_score_outputs *out)
{
    return score_loci_host(matrix, 0, m, n, params, out);
}

RB_API int rocco_score_loci_wls_f32(const float *matrix, size_t m, size_t n, const rocco_b200_score_params *params,
                                    rocco_b200_score_outputs *out)
{
    return score_loci_host(matrix, 1, m, n, params, out);
}

RB_API int rocco_crossfit_whittaker_baseline_matrix_f64(const double *matrix_values, size_t row_count, size_t column_count,
                                                        double penalty_lambda, double *baseline_out)
{
    if (!matrix_values || !baseline_out) return ST_NOMEM;
    if (row_count == 0 || column_count == 0) return 0;
    RB_TRY(ensure_device());
    HostScope lease;
    cudaStream_t st = lease.stream();
    Arena ar(st);
    double *d_in = nullptr, *d_out = nullptr;
    const size_t total = row_count * column_count;
    RB_TRY(ar.alloc(&d_in, total));
    RB_TRY(ar.alloc(&d_out, total));
    RB_CUDA(cudaMemcpyAsync(d_in, matrix_values, total * sizeof(double), cudaMemcpyHostToDevice, st));
    RB_TRY(rocco_b200_crossfit_baseline_dev(d_in, row_count, column_count, penalty_lambda, d_out, st));
    RB_CUDA(cudaMemcpyAsync(baseline_out, d_out, total * sizeof(double), cudaMemcpyDeviceToHost, st));
    RB_CUDA(cudaStreamSynchronize(st));
    return 0;
}

RB_API int rocco_crossfit_whittaker_baseline_f64(const double *y_values, size_t value_count, double penalty_lambda,
                                                 double *baseline_out)
{
    return rocco_crossfit_whittaker_baseline_matrix_f64(y_values, 1, value_count, penalty_lambda, baseline_out);
}

RB_API int rocco_score_centered_wls_f64(
    const double *centered_matrix, size_t sample_count, size_t locus_count, double lower_bound_z, double prior_df,
    double min_effect, int use_min_effect, int spatial_window, double precision_floor_ratio, double *mean_out,
    double *raw_variance_out, double *prior_variance_out, double *moderated_variance_out, double *standard_error_out,
    double *scores_out, double *degrees_of_freedom_out, int *resolved_window_out)
{
    // argument checks and status codes of wls_backend.c:779-788
    if (!centered_matrix || !mean_out || !raw_variance_out || !prior_variance_out || !moderated_variance_out ||
        !standard_error_out || !scores_out)
        return ST_INVALID;
    if (sample_count == 0 || locus_count == 0) return ST_INVALID;
    RB_TRY(ensure_device());
    HostScope lease;
    cudaStream_t st = lease.stream();
    Arena ar(st);
    double *d_c = nullptr;
    const size_t total = sample_count * locus_count;
    RB_TRY(ar.alloc(&d_c, total));
    RB_CUDA(cudaMemcpyAsync(d_c, centered_matrix, total * sizeof(double), cudaMemcpyHostToDevice, st));
    rocco_b200_score_params prm;
    rocco_b200_default_score_params(&prm);
    prm.lower_bound_z = lower_bound_z; prm.prior_df = prior_df; prm.min_effect = min_effect;
    prm.use_min_effect = use_min_effect; prm.spatial_window = spatial_window; prm.precision_floor_ratio = precision_floor_ratio;
    rocco_b200_score_outputs host{}, dev{};
    host.scores = scores_out; host.mean = mean_out; host.raw_variance = raw_variance_out;
    host.prior_variance = prior_variance_out; host.moderated_variance = moderated_variance_out;
    host.standard_error = standard_error_out;
    HostOuts ho;
    RB_TRY(run_host_outputs(ar, locus_count, host, dev, ho));
    int s = score::centered_wls(d_c, (long long)sample_count, (long long)locus_count, prm, &dev, st);
    if (s != 0) return s;
    if (degrees_of_freedom_out) *degrees_of_freedom_out = dev.total_df;
    if (resolved_window_out) *resolved_window_out = dev.resolved_spatial_window;
    return copy_back(locus_count, ho, st);
}
