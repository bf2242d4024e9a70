// Column-wise statistics over the sample axis of a [samples, bins] matrix.
//
// Replaces /root/reference/rocco/rocco.py:243-304 (score_central_tendency_chrom: np.median /
// np.quantile(method="nearest") / scipy.stats.tmean in a Python loop over bins / np.mean) and
// rocco.py:307-355 (score_dispersion_chrom: scipy median_abs_deviation / iqr / np.std / tstd).
//
// Up to a crossover in m (tile_from), one thread per bin.  Loads are coalesced along the bin axis (thread j reads X[i, j] for every sample i).  Median,
// nearest-rank quantile, MAD and IQR read one to four ranks of the column: the thread keeps just the smallest (and / or
// largest) values needed to reach them in a short sorted list in shared memory, [slot][thread] (conflict-free)
// (k_colstat_ranks).  Trimmed mean / std need the whole column: it is insertion-sorted in shared memory (k_colstat).
// All order statistics are exact.  Sums follow NumPy's own association order -- sequential over rows for axis-0
// reductions of a C-contiguous matrix, pairwise (8 accumulators, blocks of 128) for the 1-D reductions that
// scipy's tmean/tstd perform per column -- so means and standard deviations reproduce the reference's bits.
// From the crossover on, and for every m those kernels cannot hold, k_colstat_tile stages a tile of bins x all samples in
// shared memory and radix-selects each wanted rank with the whole CTA; MEAN / STD run k_colstat without shared memory.
#include "common.cuh"
#include "select.cuh"

#include <math.h>

#include <algorithm>

namespace rb {
namespace colstats {

struct Params {
    const void *x; double *out;
    long long m, n;
    int in_f32, stat;
    double arg0, arg1, power;
    int tb;
};

__device__ __forceinline__ double ldx(const Params &P, long long i, long long j)
{
    return P.in_f32 ? (double)reinterpret_cast<const float *>(P.x)[i * P.n + j]
                    : reinterpret_cast<const double *>(P.x)[i * P.n + j];
}

// np.around: round half to even
__device__ __forceinline__ long long round_half_even(double v) { return (long long)rint(v); }

// numpy pairwise sum (DOUBLE_pairwise_sum: n < 8 serial, <= 128 eight accumulators, else split in halves rounded to
// a multiple of 8) of the strided vector v[0], v[stride], ...; `sq_mean` != nullptr sums (v - *sq_mean)^2 instead.
__device__ double np_pairwise_block(const double *v, int stride, long long cnt, const double *sq_mean)
{
    auto at = [&](long long i) {
        const double x = v[i * stride];
        if (!sq_mean) return x;
        const double d = __dsub_rn(x, *sq_mean);
        return __dmul_rn(d, d);
    };
    if (cnt < 8) {
        double r = 0.0;
        for (long long i = 0; i < cnt; ++i) r = __dadd_rn(r, at(i));
        return r;
    }
    double r[8];
    for (int k = 0; k < 8; ++k) r[k] = at(k);
    long long i = 8;
    for (; i < cnt - (cnt % 8); i += 8)
        for (int k = 0; k < 8; ++k) r[k] = __dadd_rn(r[k], at(i + k));
    double res = __dadd_rn(__dadd_rn(__dadd_rn(r[0], r[1]), __dadd_rn(r[2], r[3])),
                           __dadd_rn(__dadd_rn(r[4], r[5]), __dadd_rn(r[6], r[7])));
    for (; i < cnt; ++i) res = __dadd_rn(res, at(i));
    return res;
}

__device__ double np_pairwise(const double *v, int stride, long long cnt, const double *sq_mean)
{
    // explicit post-order walk of numpy's recursion (depth <= 8 for any supported sample count)
    struct Frame { long long lo, cnt; int state; double left; };
    Frame st[12];
    int sp = 0;
    st[0] = Frame{0, cnt, 0, 0.0};
    double ret = 0.0;
    while (sp >= 0) {
        Frame &f = st[sp];
        if (f.cnt <= 128) { ret = np_pairwise_block(v + f.lo * stride, stride, f.cnt, sq_mean); --sp; continue; }
        long long n2 = f.cnt / 2;
        n2 -= n2 % 8;
        if (f.state == 0) { f.state = 1; st[sp + 1] = Frame{f.lo, n2, 0, 0.0}; ++sp; }
        else if (f.state == 1) { f.left = ret; f.state = 2; st[sp + 1] = Frame{f.lo + n2, f.cnt - n2, 0, 0.0}; ++sp; }
        else { ret = __dadd_rn(f.left, ret); --sp; }
    }
    return ret;
}

// np.power(x, scalar): NumPy's scalar fast paths (square, sqrt, reciprocal) are exact; libm pow otherwise
__device__ __forceinline__ double np_power(double x, double p)
{
    if (p == 1.0) return x;
    if (p == 2.0) return __dmul_rn(x, x);
    if (p == 0.5) return sqrt(x);
    if (p == -1.0) return 1.0 / x;
    if (p == 0.0) return 1.0;
    return pow(x, p);
}

__device__ __forceinline__ double lerp_np(double a, double b, double t)
{
    const double d = __dsub_rn(b, a);
    return (t >= 0.5) ? __dsub_rn(b, __dmul_rn(d, __dsub_rn(1.0, t))) : __dadd_rn(a, __dmul_rn(d, t));
}

__global__ void k_colstat(Params P)
{
    extern __shared__ double s_col[];                 // [m][tb]
    const int tb = P.tb;
    const long long j = (long long)blockIdx.x * tb + threadIdx.x;
    if (j >= P.n) return;
    const long long m = P.m;
    double *col = s_col + threadIdx.x;
    auto S = [&](long long i) -> double & { return col[i * tb]; };

    double result = 0.0;
    const int stat = P.stat;
    if (stat == ROCCO_STAT_MEAN || stat == ROCCO_STAT_STD) {
        // axis-0 reduction of a C-contiguous matrix: rows are added one after the other
        double sum = ldx(P, 0, j);
        for (long long i = 1; i < m; ++i) sum = __dadd_rn(sum, ldx(P, i, j));
        const double mean = sum / (double)m;
        if (stat == ROCCO_STAT_MEAN) result = mean;
        else {
            double d0 = __dsub_rn(ldx(P, 0, j), mean);
            double ss = __dmul_rn(d0, d0);
            for (long long i = 1; i < m; ++i) { const double d = __dsub_rn(ldx(P, i, j), mean); ss = __dadd_rn(ss, __dmul_rn(d, d)); }
            result = sqrt(ss / (double)m);
        }
    } else {
        // insertion sort of the column in shared memory
        for (long long i = 0; i < m; ++i) {
            const double v = ldx(P, i, j);
            long long q = i;
            while (q > 0 && S(q - 1) > v) { S(q) = S(q - 1); --q; }
            S(q) = v;
        }
        {                                                      // TMEAN / TSTD: nearest-rank limits, inclusive (the rank-only modes run in k_colstat_ranks)
            long long kl = round_half_even((double)(m - 1) * P.arg0);
            long long kh = round_half_even((double)(m - 1) * (1.0 - P.arg0));
            kl = kl < 0 ? 0 : (kl >= m ? m - 1 : kl);
            kh = kh < 0 ? 0 : (kh >= m ? m - 1 : kh);
            const double lim_lo = S(kl), lim_hi = S(kh);
            long long cnt = 0;
            for (long long i = 0; i < m; ++i) { const double v = ldx(P, i, j); cnt += (v >= lim_lo && v <= lim_hi); }
            if (stat == ROCCO_STAT_TMEAN) {
                // scipy.stats.tmean: sum over the column in row order with outsiders replaced by 0, / count
                for (long long i = 0; i < m; ++i) { const double v = ldx(P, i, j); S(i) = (v >= lim_lo && v <= lim_hi) ? v : 0.0; }
                result = cnt > 0 ? np_pairwise(col, tb, m, nullptr) / (double)cnt : NAN;
            } else {
                // sample standard deviation (ddof 1) of the kept values (np.std on the compressed 1-D vector):
                // kept values are gathered in row order into the (now free) shared column
                long long k = 0;
                for (long long i = 0; i < m; ++i) { const double v = ldx(P, i, j); if (v >= lim_lo && v <= lim_hi) S(k++) = v; }
                const double mean = np_pairwise(col, tb, cnt, nullptr) / (double)cnt;
                result = cnt > 1 ? sqrt(np_pairwise(col, tb, cnt, &mean) / (double)(cnt - 1)) : NAN;
            }
        }
    }
    P.out[j] = np_power(result, P.power);
}

// ---- order statistics that need only a few ranks: MEDIAN, QUANTILE, MAD, IQR
// Instead of sorting the whole column, a thread keeps the `cap` smallest (ascending list) and / or the `cap` largest
// (descending list) values seen so far -- half the shared memory per column (twice the resident warps) and fewer than half
// the compare-and-shift steps for a median.  Lists live in shared memory as [slot][thread] (conflict-free).
struct PartialLists { int cap_lo, cap_hi; };

template <bool SMALLEST>
__device__ __forceinline__ void partial_insert(double *L, int tb, int cap, int &len, double v)
{
    auto before = [](double a, double b) { return SMALLEST ? a < b : a > b; };      // a sorts before b
    if (len == cap) {
        if (!before(v, L[(cap - 1) * tb])) return;       // not among the kept ones
        --len;                                           // the last kept value drops out
    }
    int q = len;
    while (q > 0 && before(v, L[(q - 1) * tb])) { L[q * tb] = L[(q - 1) * tb]; --q; }
    L[q * tb] = v;
    ++len;
}

__global__ void k_colstat_ranks(Params P, PartialLists C)
{
    extern __shared__ double s_col[];                 // [cap_lo + cap_hi][tb]
    const int tb = P.tb;
    const long long j = (long long)blockIdx.x * tb + threadIdx.x;
    if (j >= P.n) return;
    const long long m = P.m;
    double *lo = s_col + threadIdx.x;                 // ascending: the cap_lo smallest
    double *hi = s_col + (size_t)C.cap_lo * tb + threadIdx.x;      // descending: the cap_hi largest
    int nlo = 0, nhi = 0;
    for (long long i = 0; i < m; ++i) {
        const double v = ldx(P, i, j);
        if (C.cap_lo) partial_insert<true>(lo, tb, C.cap_lo, nlo, v);
        if (C.cap_hi) partial_insert<false>(hi, tb, C.cap_hi, nhi, v);
    }
    // ascending rank r of the column (the caller sized the lists so that every rank asked for is covered)
    auto rank = [&](long long r) { return r < C.cap_lo ? lo[r * tb] : hi[(m - 1 - r) * tb]; };
    auto median_of = [&]() { return (m & 1) ? rank(m / 2) : __dadd_rn(rank(m / 2 - 1), rank(m / 2)) / 2.0; };
    double result = 0.0;
    const int stat = P.stat;
    if (stat == ROCCO_STAT_MEDIAN) {
        result = median_of();
    } else if (stat == ROCCO_STAT_QUANTILE) {
        long long k = round_half_even((double)(m - 1) * P.arg0);
        k = k < 0 ? 0 : (k >= m ? m - 1 : k);
        result = rank(k);
    } else if (stat == ROCCO_STAT_MAD) {
        const double med = median_of();
        nlo = 0;                                       // second pass: the smallest |x - med| (same list, same capacity)
        for (long long i = 0; i < m; ++i) partial_insert<true>(lo, tb, C.cap_lo, nlo, fabs(__dsub_rn(ldx(P, i, j), med)));
        result = median_of();
    } else {                                           // IQR (scipy.stats.iqr, linear interpolation)
        double pv[2];
        for (int k = 0; k < 2; ++k) {
            const double q = (k == 0 ? P.arg0 : P.arg1) / 100.0;
            const double vi = (double)(m - 1) * q;
            double prev = floor(vi);
            long long ip = (long long)prev, in = ip + 1;
            if (vi >= (double)(m - 1)) { ip = m - 1; in = m - 1; }
            if (vi < 0) { ip = 0; in = 0; }
            const double gamma = __dsub_rn(vi, prev);
            pv[k] = lerp_np(rank(ip), rank(in), gamma);
        }
        result = __dsub_rn(pv[1], pv[0]);
    }
    P.out[j] = np_power(result, P.power);
}

// ---- any sample count: k_colstat_tile
// A CTA stages W consecutive bins x all m rows in shared memory, each value read from HBM once, as order-preserving
// 64-bit keys (sign-flip; -0.0 and +0.0 share one key, as they compare equal in NumPy), column c contiguous in row order
// at tile + c * ld (ld odd: the staging stores of one warp spread over the banks).  The wanted ranks of a column come from
// score::block_select over the whole CTA, one column after the other; a rank already covered by the previous select's
// run of equal keys costs nothing.  TMEAN / TSTD then sum each column in row order with np_pairwise, one thread per column.
// Results are the bits of k_colstat / k_colstat_ranks wherever those run (up to the sign of a zero result).
constexpr int TILE_THREADS = 256, TILE_MAX_W = 32;

__device__ __forceinline__ unsigned long long dkey(double v)
{
    const unsigned long long b = (unsigned long long)__double_as_longlong(__dadd_rn(v, 0.0));     // -0.0 -> +0.0
    return (b >> 63) ? ~b : (b | 0x8000000000000000ULL);
}

__device__ __forceinline__ double dval(unsigned long long k)
{
    return __longlong_as_double((long long)((k >> 63) ? (k & 0x7fffffffffffffffULL) : ~k));
}

struct RankCache { unsigned long long key; int below, equal; };

// key of 0-based ascending rank r of the column (uniform over the CTA)
__device__ __forceinline__ unsigned long long rank_key(const unsigned long long *col, int m, long long r, score::SelScratch &S,
                                                       RankCache &rc)
{
    if (rc.equal > 0 && r >= rc.below && r < (long long)rc.below + rc.equal) return rc.key;
    rc.key = score::block_select<TILE_THREADS, true>(col, m, (int)r, nullptr, 0ULL, S, &rc.below, &rc.equal);
    return rc.key;
}

__global__ void __launch_bounds__(TILE_THREADS, 2) k_colstat_tile(Params P, int lw, int ld)
{
    extern __shared__ unsigned long long s_dyn[];          // SelScratch, then the [W][ld] key tile
    __shared__ unsigned long long s_lim[2][TILE_MAX_W];     // TMEAN / TSTD: the limit keys of each column
    score::SelScratch &S = score::plan_scratch(s_dyn);
    unsigned long long *tile = s_dyn + sizeof(score::SelScratch) / sizeof(unsigned long long);
    const int W = 1 << lw;
    const long long j0 = (long long)blockIdx.x * W;
    const int w = (int)min((long long)W, P.n - j0);
    const int m = (int)P.m;
    {                                                       // stage: a warp reads 32 / W rows of W consecutive bins
        const int c = threadIdx.x & (W - 1), step = TILE_THREADS >> lw;
        if (c < w) {
            unsigned long long *col = tile + (size_t)c * ld;
            if (P.in_f32) {
                const float *x = reinterpret_cast<const float *>(P.x) + j0 + c;
#pragma unroll 4
                for (int i = threadIdx.x >> lw; i < m; i += step) col[i] = dkey((double)x[(long long)i * P.n]);
            } else {
                const double *x = reinterpret_cast<const double *>(P.x) + j0 + c;
#pragma unroll 4
                for (int i = threadIdx.x >> lw; i < m; i += step) col[i] = dkey(x[(long long)i * P.n]);
            }
        }
    }
    __syncthreads();
    // the ranks each column needs (the same for every column): median / MAD 0-1, quantile 0, IQR 0-3, TMEAN / TSTD 0-1
    const int stat = P.stat;
    long long want[4];
    double gam[2] = {0.0, 0.0};
    int nw;
    if (stat == ROCCO_STAT_MEDIAN || stat == ROCCO_STAT_MAD) {
        want[0] = (m & 1) ? m / 2 : m / 2 - 1; want[1] = m / 2; nw = 2;
    } else if (stat == ROCCO_STAT_QUANTILE) {
        long long k = round_half_even((double)(m - 1) * P.arg0);
        want[0] = k < 0 ? 0 : (k >= m ? m - 1 : k); nw = 1;
    } else if (stat == ROCCO_STAT_IQR) {                   // scipy.stats.iqr, linear interpolation
        for (int k = 0; k < 2; ++k) {
            const double q = (k == 0 ? P.arg0 : P.arg1) / 100.0;
            const double vi = (double)(m - 1) * q;
            double prev = floor(vi);
            long long ip = (long long)prev, in = ip + 1;
            if (vi >= (double)(m - 1)) { ip = m - 1; in = m - 1; }
            if (vi < 0) { ip = 0; in = 0; }
            gam[k] = __dsub_rn(vi, prev);
            want[2 * k] = ip; want[2 * k + 1] = in;
        }
        nw = 4;
    } else {                                               // TMEAN / TSTD: nearest-rank limits, inclusive
        long long kl = round_half_even((double)(m - 1) * P.arg0);
        long long kh = round_half_even((double)(m - 1) * (1.0 - P.arg0));
        want[0] = kl < 0 ? 0 : (kl >= m ? m - 1 : kl);
        want[1] = kh < 0 ? 0 : (kh >= m ? m - 1 : kh);
        nw = 2;
    }
    for (int c = 0; c < w; ++c) {
        unsigned long long *col = tile + (size_t)c * ld;
        unsigned long long key[4];
        for (int pass = 0;; ++pass) {
            RankCache rc{0ULL, 0, 0};
#pragma unroll 1
            for (int q = 0; q < nw; ++q) key[q] = rank_key(col, m, want[q], S, rc);
            if (stat != ROCCO_STAT_MAD || pass == 1) break;
            // MAD: the same ranks of |x - median|, rewritten in place
            const double med = __dadd_rn(dval(key[0]), dval(key[1])) / 2.0;
            const double mid = (m & 1) ? dval(key[1]) : med;
            for (int i = threadIdx.x; i < m; i += TILE_THREADS) col[i] = dkey(fabs(__dsub_rn(dval(col[i]), mid)));
            __syncthreads();
        }
        double result;
        if (stat == ROCCO_STAT_MEDIAN || stat == ROCCO_STAT_MAD)
            result = (m & 1) ? dval(key[1]) : __dadd_rn(dval(key[0]), dval(key[1])) / 2.0;
        else if (stat == ROCCO_STAT_QUANTILE)
            result = dval(key[0]);
        else if (stat == ROCCO_STAT_IQR)
            result = __dsub_rn(lerp_np(dval(key[2]), dval(key[3]), gam[1]), lerp_np(dval(key[0]), dval(key[1]), gam[0]));
        else {
            if (threadIdx.x == 0) { s_lim[0][c] = key[0]; s_lim[1][c] = key[1]; }
            continue;
        }
        if (threadIdx.x == 0) P.out[j0 + c] = np_power(result, P.power);
    }
    if (stat != ROCCO_STAT_TMEAN && stat != ROCCO_STAT_TSTD) return;
    __syncthreads();
    const int c = threadIdx.x;
    if (c >= w) return;
    unsigned long long *colk = tile + (size_t)c * ld;
    double *col = reinterpret_cast<double *>(colk);        // rewritten in place as the doubles that are summed
    const unsigned long long klo = s_lim[0][c], khi = s_lim[1][c];
    long long cnt = 0;
    double result;
    if (stat == ROCCO_STAT_TMEAN) {
        // scipy.stats.tmean: sum over the column in row order with outsiders replaced by 0, / count
        for (int i = 0; i < m; ++i) {
            const unsigned long long k = colk[i];
            const bool keep = k >= klo && k <= khi;
            cnt += keep;
            col[i] = keep ? dval(k) : 0.0;
        }
        result = cnt > 0 ? np_pairwise(col, 1, m, nullptr) / (double)cnt : NAN;
    } else {
        // np.std(ddof=1) of the kept values gathered in row order (write index <= read index)
        for (int i = 0; i < m; ++i) {
            const unsigned long long k = colk[i];
            if (k >= klo && k <= khi) col[cnt++] = dval(k);
        }
        const double mean = np_pairwise(col, 1, cnt, nullptr) / (double)cnt;
        result = cnt > 1 ? sqrt(np_pairwise(col, 1, cnt, &mean) / (double)(cnt - 1)) : NAN;
    }
    P.out[j0 + c] = np_power(result, P.power);
}

// largest m whose one-column tile fits in a CTA's shared memory
static size_t tile_max_m(int smem_optin)
{
    const size_t avail = (size_t)smem_optin - sizeof(score::SelScratch) - 2 * TILE_MAX_W * sizeof(unsigned long long);
    const size_t ld = avail / sizeof(unsigned long long);
    return (ld & 1) ? ld : ld - 1;                         // ld = m | 1
}

static int run_tile(const Params &P0, cudaStream_t st)
{
    Params P = P0;
    const size_t m = (size_t)P.m, n = (size_t)P.n;
    int dev = 0, optin = 0;
    RB_CUDA(cudaGetDevice(&dev));
    RB_CUDA(cudaDeviceGetAttribute(&optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev));
    const size_t max_m = tile_max_m(optin);
    if (m > max_m) {
        set_error("column statistics support at most %zu samples (one column of 64-bit keys in shared memory)", max_m);
        return ST_INVALID;
    }
    const size_t ld = m | 1, col_bytes = ld * sizeof(unsigned long long), base = sizeof(score::SelScratch);
    const size_t limit = (size_t)optin - 2 * TILE_MAX_W * sizeof(unsigned long long);
    // widest power of two <= 32 within 100 KB (two CTAs per SM, which is what the registers allow), but at least a 32-byte
    // sector of every row segment (8 float32 / 4 float64 bins) when that fits at all
    const int sector_w = P.in_f32 ? 8 : 4;
    int lw = 5;
    while (lw > 0 && base + ((size_t)1 << lw) * col_bytes > 100 * 1024) --lw;
    while ((1 << lw) < sector_w && base + ((size_t)2 << lw) * col_bytes <= limit) ++lw;
    const int W = 1 << lw;
    const size_t smem = base + (size_t)W * col_bytes;
    RB_CUDA(cudaFuncSetAttribute(k_colstat_tile, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)limit));
    RB_PROF("k_colstat_tile", st, (double)m * n * (P.in_f32 ? 4.0 : 8.0) + 8.0 * n);
    k_colstat_tile<<<(unsigned)((n + W - 1) / W), TILE_THREADS, smem, st>>>(P, lw, (int)ld);
    RB_LAUNCH_CHECK();
    return 0;
}

// 1: k_colstat_tile for every m >= 2 (tests compare it with the other kernels); anything else: chosen from m and the statistic
static std::atomic<int> g_colstat_mode{0};

// smallest m at which k_colstat_tile takes a statistic in automatic mode even where the list kernels fit.  Until
// tools/colstat_large.py has measured a crossover the list kernels keep every size they can hold (DESIGN.md section 3).
static size_t tile_from(int stat, int in_f32)
{
    (void)stat; (void)in_f32;
    return (size_t)1 << 62;
}

__global__ void k_single_row(Params P)
{
    // m == 1: central tendency = row ** power; dispersion = zeros ** power (rocco.py:254-255, 318-319)
    const long long j = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= P.n) return;
    const bool dispersion = P.stat >= ROCCO_STAT_MAD;
    const double v = dispersion ? 0.0 : ldx(P, 0, j);
    P.out[j] = np_power(v, P.power);
}

// MEAN / STD read the matrix only: k_colstat without the per-column shared-memory reservation serves any m
static int run_moments(Params P, cudaStream_t st)
{
    P.tb = 128;
    RB_PROF("k_colstat", st, (double)P.m * P.n * (P.in_f32 ? 4.0 : 8.0) + 8.0 * P.n);
    k_colstat<<<(unsigned)((P.n + 127) / 128), 128, 0, st>>>(P);
    RB_LAUNCH_CHECK();
    return 0;
}

static int run(const void *d_x, int dtype, size_t m, size_t n, int stat, double arg0, double arg1, double power,
               double *d_out, cudaStream_t st)
{
    if (!d_x || !d_out || m == 0 || n == 0) return ST_INVALID;
    if (stat < ROCCO_STAT_MEDIAN || stat > ROCCO_STAT_TSTD || (dtype != 0 && dtype != 1)) return ST_INVALID;
    RB_TRY(ensure_device());
    Params P{};
    P.x = d_x; P.out = d_out; P.m = (long long)m; P.n = (long long)n; P.in_f32 = dtype; P.stat = stat;
    P.arg0 = arg0; P.arg1 = arg1; P.power = power;
    if (m == 1) {
        k_single_row<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(P);
        RB_LAUNCH_CHECK();
        return 0;
    }
    const bool moments = stat == ROCCO_STAT_MEAN || stat == ROCCO_STAT_STD;
    if (g_colstat_mode.load() == 1 || m >= tile_from(stat, dtype)) return moments ? run_moments(P, st) : run_tile(P, st);
    // ranks wanted by the order-statistic modes -> list capacities (ascending ranks below cap_lo, the rest from the top)
    if (stat == ROCCO_STAT_MEDIAN || stat == ROCCO_STAT_QUANTILE || stat == ROCCO_STAT_MAD || stat == ROCCO_STAT_IQR) {
        long long r_min = 0, r_max = 0;                    // smallest and largest 0-based rank read
        const long long mm = (long long)m;
        auto clampr = [&](long long r) { return r < 0 ? 0 : (r >= mm ? mm - 1 : r); };
        if (stat == ROCCO_STAT_MEDIAN || stat == ROCCO_STAT_MAD) { r_min = (mm & 1) ? mm / 2 : mm / 2 - 1; r_max = mm / 2; }
        else if (stat == ROCCO_STAT_QUANTILE) { r_min = r_max = clampr((long long)nearbyint((double)(mm - 1) * arg0)); }
        else {
            long long lo_r = mm, hi_r = -1;
            for (int k = 0; k < 2; ++k) {
                const double vi = (double)(mm - 1) * ((k == 0 ? arg0 : arg1) / 100.0);
                long long ip = (long long)floor(vi), in = ip + 1;
                if (vi >= (double)(mm - 1)) { ip = mm - 1; in = mm - 1; }
                if (vi < 0) { ip = 0; in = 0; }
                lo_r = std::min(lo_r, std::min(clampr(ip), clampr(in))); hi_r = std::max(hi_r, std::max(clampr(ip), clampr(in)));
            }
            r_min = lo_r; r_max = hi_r;
        }
        // one ascending list up to r_max, or one descending list down to r_min, or both split at the middle -- whichever is smallest
        PartialLists C{};
        const long long only_lo = r_max + 1, only_hi = mm - r_min;
        long long split = only_lo;                          // ranks < mm/2+1 from the bottom, the others from the top
        if (stat == ROCCO_STAT_IQR) {
            // two rank pairs: the lower pair from the bottom, the upper pair from the top
            long long pair_hi[2], pair_lo[2];
            for (int k = 0; k < 2; ++k) {
                const double vi = (double)(mm - 1) * ((k == 0 ? arg0 : arg1) / 100.0);
                long long ip = (long long)floor(vi), in = ip + 1;
                if (vi >= (double)(mm - 1)) { ip = mm - 1; in = mm - 1; }
                if (vi < 0) { ip = 0; in = 0; }
                pair_lo[k] = clampr(std::min(ip, in)); pair_hi[k] = clampr(std::max(ip, in));
            }
            const int a = pair_hi[0] <= pair_hi[1] ? 0 : 1, b = 1 - a;      // a: the lower percentile
            const long long both = (pair_hi[a] + 1) + (mm - pair_lo[b]);
            if (both < std::min(only_lo, only_hi) && pair_hi[a] + 1 <= pair_lo[b]) { C.cap_lo = (int)(pair_hi[a] + 1); C.cap_hi = (int)(mm - pair_lo[b]); split = -1; }
        }
        if (split >= 0) {
            if (stat == ROCCO_STAT_MAD || only_lo <= only_hi) { C.cap_lo = (int)only_lo; C.cap_hi = 0; }     // (MAD reuses the ascending list)
            else { C.cap_lo = 0; C.cap_hi = (int)only_hi; }
        }
        const size_t slots = (size_t)C.cap_lo + (size_t)C.cap_hi;
        const size_t budget_r = 200 * 1024;
        int tbr = 128;
        while (tbr > 32 && slots * tbr * 8 > budget_r) tbr -= 32;
        if (slots * tbr * 8 > budget_r) return run_tile(P, st);            // the lists do not fit: no list kernel
        P.tb = tbr;
        const size_t smem_r = slots * tbr * sizeof(double);
        RB_CUDA(cudaFuncSetAttribute(k_colstat_ranks, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)budget_r));
        RB_PROF("k_colstat", st, (double)m * n * (dtype ? 4.0 : 8.0) + 8.0 * n);
        k_colstat_ranks<<<(unsigned)((n + tbr - 1) / tbr), tbr, smem_r, st>>>(P, C);
        RB_LAUNCH_CHECK();
        return 0;
    }
    const size_t budget = 192 * 1024;
    int tb = (int)std::min<size_t>(128, budget / (8 * m));
    tb = (tb / 32) * 32;
    if (tb < 32) return moments ? run_moments(P, st) : run_tile(P, st);     // the column does not fit
    P.tb = tb;
    const size_t smem = (size_t)tb * m * sizeof(double);
    RB_CUDA(cudaFuncSetAttribute(k_colstat, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)budget));
    RB_PROF("k_colstat", st, (double)m * n * (dtype ? 4.0 : 8.0) + 8.0 * n);
    k_colstat<<<(unsigned)((n + tb - 1) / tb), tb, smem, st>>>(P);
    RB_LAUNCH_CHECK();
    return 0;
}

}  // namespace colstats
}  // namespace rb

using namespace rb;
#define RB_API extern "C" __attribute__((visibility("default")))

RB_API int rocco_b200_column_stat_dev(const void *d_matrix, int dtype, size_t m, size_t n, int stat, double arg0, double arg1,
                                      double power, double *d_out, void *cuda_stream)
{
    return colstats::run(d_matrix, dtype, m, n, stat, arg0, arg1, power, d_out, (cudaStream_t)cuda_stream);
}

RB_API int rocco_b200_colstat_set_mode(int mode)
{
    return colstats::g_colstat_mode.exchange(mode == 1 ? 1 : 0);
}

RB_API int rocco_column_stat_f64(const double *matrix, size_t m, size_t n, int stat, double arg0, double arg1, double power,
                                 double *out)
{
    if (!matrix || !out || m == 0 || n == 0) return ST_INVALID;
    RB_TRY(ensure_device());
    HostScope lease;
    cudaStream_t st = lease.stream();
    Arena ar(st);
    double *d_x = nullptr, *d_o = nullptr;
    RB_TRY(ar.alloc(&d_x, m * n));
    RB_TRY(ar.alloc(&d_o, n));
    RB_CUDA(cudaMemcpyAsync(d_x, matrix, m * n * sizeof(double), cudaMemcpyHostToDevice, st));
    RB_TRY(colstats::run(d_x, 0, m, n, stat, arg0, arg1, power, d_o, st));
    RB_CUDA(cudaMemcpyAsync(out, d_o, n * sizeof(double), cudaMemcpyDeviceToHost, st));
    RB_CUDA(cudaStreamSynchronize(st));
    return 0;
}
