// Dependent-wild-bootstrap budget null and the statistics either side of it (SURVEY.md 8(f) ranks 1-2).
//
// Replaces, device-resident, /root/reference/rocco/inference.py:446-501 (effective sample size), 533-570 (Bartlett
// multiplier field), 638-681 (one bootstrap draw), 684-716 (null residual template), 719-985 (the draw loop with its
// adaptive stop), 988-1148 (observed-vs-null summary) and rocco.py:751-789 (median of the positive scores for the
// automatic gamma).  Every draw re-runs the centred-WLS scoring chain of wls.cu / trend.cu on  template x weights.
//
// Random streams: the reference draws NumPy PCG64 normals (one generator per draw, samples in order).  By default the
// innovations here are counter-based -- Philox4x32-10 keyed by the seed, counter = (pair index, sample, draw) ->
// Box-Muller in double -- so a draw is reproducible and independent of tiling, but the streams differ from NumPy's:
// parity with the reference is statistical.  With random_streams = 1 the reference's own streams are generated on the
// device (numpy_streams.cu) in groups of rows, and the FIR reads them exactly as it reads supplied innovations: the
// field is then the reference's.  The caller may also pass the innovations themselves (`d_innovations`), which is how
// tests replay the reference's own streams through these kernels.
//
// Sample sharding: the estimator also runs with the samples split over ranks (the layout of the sample-sharded scoring).
// Everything per sample -- the template, the multiplier field (row r of a shard draws the stream of global sample
// sample_offset + r), the per-row WLS stages -- stays on the rank; the only cross-sample step of a scoring pass, the column
// sums of the combine, goes through the caller's all-reduce (2n sums + status slots); everything after a score track exists
// (sort, centre/scale, track sums, adaptive stop, ESS, positive median) is recomputed by every rank from the bit-identical
// reduced track.  Every decision taken after a reduce depends only on reduced data, and a rank-local failure is carried to
// the next reduce in the status slots, so all ranks leave together with the same status.
#include <cub/cub.cuh>

#include <cmath>

#include "common.cuh"
#include "numpy_streams.cuh"
#include "score.cuh"

namespace rb {
namespace budget {

constexpr int FIR_THREADS = 512;
constexpr int FIR_ITEMS = 16;
constexpr int FIR_T = FIR_THREADS * FIR_ITEMS;        // outputs per CTA
constexpr int MAX_BANDWIDTH = 2048;                   // taps = 2 b + 1 <= 4097 (n^(1/3) rule: 171 at 5 M bins)
constexpr int AC_T = 4096, AC_THREADS = 256, AC_MAXLAG = 4096;
constexpr int RED_BLOCKS = 1184, RED_THREADS = 256;   // 8 CTAs per SM x 148

// 16 bins per thread: position i lives at i + i/16 (thread stride 17 doubles: conflict-free 8-byte accesses)
__host__ __device__ __forceinline__ int padpos(int i) { return i + (i >> 4); }

// ------------------------------------------------------------------ Philox4x32-10 + Box-Muller
__device__ __forceinline__ uint4 philox4x32_10(uint4 c, uint2 k)
{
#pragma unroll
    for (int r = 0; r < 10; ++r) {
        const unsigned hi0 = __umulhi(0xD2511F53u, c.x), lo0 = 0xD2511F53u * c.x;
        const unsigned hi1 = __umulhi(0xCD9E8D57u, c.z), lo1 = 0xCD9E8D57u * c.z;
        c = make_uint4(hi1 ^ c.y ^ k.x, lo1, hi0 ^ c.w ^ k.y, lo0);
        k.x += 0x9E3779B9u; k.y += 0xBB67AE85u;
    }
    return c;
}

// two independent N(0,1) for (pair, sample, draw)
__device__ __forceinline__ double2 normal_pair(unsigned long long pair, unsigned sample, unsigned draw, uint2 key)
{
    const uint4 r = philox4x32_10(make_uint4((unsigned)pair, (unsigned)(pair >> 32), sample, draw), key);
    const unsigned long long a = ((unsigned long long)r.x << 21) | (r.y >> 11);       // 53 bits
    const unsigned long long b = ((unsigned long long)r.z << 21) | (r.w >> 11);
    const double u1 = ((double)a + 0.5) * 1.1102230246251565e-16;                     // (0, 1)
    const double u2 = ((double)b + 0.5) * 1.1102230246251565e-16;
    const double rad = sqrt(-2.0 * log(u1));
    double s, c;
    sincospi(2.0 * u2, &s, &c);
    return make_double2(rad * c, rad * s);
}

// ------------------------------------------------------------------ template = centered - max(mean, 0)
__global__ void __launch_bounds__(256) k_template(const double *__restrict__ C, const double *__restrict__ mean, long long m,
                                                  long long n, double *__restrict__ T)
{
    const long long total = m * n;
    for (long long g = (long long)blockIdx.x * blockDim.x + threadIdx.x; g < total; g += (long long)gridDim.x * blockDim.x) {
        const long long j = g % n;
        T[g] = C[g] - fmax(mean[j], 0.0);
    }
}

// ------------------------------------------------------------------ multiplier field: FIR of the innovations
// raw[i][j] = sum_k taps[k] * z[i][j + k],  k = 0 .. K-1, K = 2b + 1  (valid-mode correlation; the taps are symmetric, so
// this is the reference's fftconvolve(..., mode="valid")).  One CTA per (tile of FIR_T outputs, sample); the z span of
// the tile is staged in shared memory (generated in place when no innovations are supplied).  The Bartlett taps are a
// triangle, taps[k] = h * (b + 1 - |k - b|), so consecutive outputs differ by h * (R_j - L_j) with the two box sums
//   L_j = z[j] + .. + z[j+b],   R_j = z[j+b+1] + .. + z[j+2b+1]:
// every thread forms its first output (and L, R) directly -- K fused multiply-adds -- and slides the next 15, which
// keeps the rounding of a slide chain at 15 steps (~1e-15) instead of the row length.
// The Philox stream of row r is that of sample sample_offset + r: a shard's field equals those rows of the whole field.
__global__ void __launch_bounds__(FIR_THREADS, 2) k_wild_fir(const double *__restrict__ innov, long long innov_stride, uint2 key,
                                                          unsigned draw, unsigned sample_offset, long long n, int K,
                                                          const double *__restrict__ taps, double h, double *__restrict__ raw,
                                                          double2 *__restrict__ partial, int tiles)
{
    extern __shared__ double s_fir[];
    double *s_x = s_fir;                                   // padpos(FIR_T + K + 8)
    double *s_t = s_fir + padpos(FIR_T + K + 8) + 8;       // K taps
    __shared__ double2 s_red[FIR_THREADS / 32];
    const int tid = threadIdx.x;
    const long long row = blockIdx.y;
    const long long j0 = (long long)blockIdx.x * FIR_T;
    const int cnt = (int)min((long long)FIR_T, n - j0);
    const int span = cnt + K - 1;
    const int staged = FIR_T + K + 1;                      // the last slide reads z[FIR_T - 2 + K + 1]
    for (int k = tid; k < K; k += FIR_THREADS) s_t[k] = taps[k];
    if (innov) {
        const double *src = innov + row * innov_stride + j0;
        for (int e = tid; e < staged; e += FIR_THREADS) s_x[padpos(e)] = (e < span) ? src[e] : 0.0;
    } else {
        // j0 is even: pair p of this tile is global pair j0/2 + p, identical whichever tile generates it
        for (int p = tid; 2 * p < staged; p += FIR_THREADS) {
            const int e = 2 * p;
            double2 z = make_double2(0.0, 0.0);
            if (e < span) z = normal_pair((unsigned long long)(j0 / 2 + p), sample_offset + (unsigned)row, draw, key);
            s_x[padpos(e)] = z.x;
            if (e + 1 < staged) s_x[padpos(e + 1)] = (e + 1 < span) ? z.y : 0.0;
        }
    }
    __syncthreads();
    const int base = tid * FIR_ITEMS, b = (K - 1) / 2;
    double w = 0.0, L = 0.0, R = 0.0;
    for (int k = 0; k <= b; ++k) { const double z = s_x[padpos(base + k)]; w = fma(s_t[k], z, w); L += z; }
    for (int k = b + 1; k < K; ++k) { const double z = s_x[padpos(base + k)]; w = fma(s_t[k], z, w); R += z; }
    R += s_x[padpos(base + K)];
    double out[FIR_ITEMS];
    out[0] = w;
#pragma unroll
    for (int r = 1; r < FIR_ITEMS; ++r) {
        w = fma(h, R - L, w);
        out[r] = w;
        const double zj = s_x[padpos(base + r - 1)], zm = s_x[padpos(base + r + b)], ze = s_x[padpos(base + r + K)];
        L += zm - zj;
        R += ze - zm;
    }
    __syncthreads();
    double s1 = 0.0, s2 = 0.0;
#pragma unroll
    for (int r = 0; r < FIR_ITEMS; ++r) {
        const double v = (base + r < cnt) ? out[r] : 0.0;
        s_x[padpos(base + r)] = v;
        s1 += v; s2 = fma(v, v, s2);
    }
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) { s1 += __shfl_down_sync(0xffffffffu, s1, d); s2 += __shfl_down_sync(0xffffffffu, s2, d); }
    if ((tid & 31) == 0) s_red[tid >> 5] = make_double2(s1, s2);
    __syncthreads();
    if (tid == 0) {
        double a = 0.0, c = 0.0;
        for (int q = 0; q < FIR_THREADS / 32; ++q) { a += s_red[q].x; c += s_red[q].y; }
        partial[row * tiles + blockIdx.x] = make_double2(a, c);
    }
    double *dst = raw + row * n + j0;
    for (int e = tid; e < cnt; e += FIR_THREADS) dst[e] = s_x[padpos(e)];
}

// per-sample mean and population s.d. of the raw field, partials added in tile order (deterministic)
__global__ void __launch_bounds__(256) k_row_moments(const double2 *__restrict__ partial, int tiles, long long n, double2 *stats,
                                                     int *bad)
{
    __shared__ double2 s[256];
    const long long row = blockIdx.x;
    double a = 0.0, b = 0.0;
    for (int t = threadIdx.x; t < tiles; t += 256) { const double2 p = partial[row * tiles + t]; a += p.x; b += p.y; }
    s[threadIdx.x] = make_double2(a, b);
    __syncthreads();
    for (int d = 128; d > 0; d >>= 1) {
        if (threadIdx.x < d) { s[threadIdx.x].x += s[threadIdx.x + d].x; s[threadIdx.x].y += s[threadIdx.x + d].y; }
        __syncthreads();
    }
    if (threadIdx.x == 0) {
        const double mean = s[0].x / (double)n;
        const double var = fmax(s[0].y / (double)n - mean * mean, 0.0);
        const double sd = sqrt(var);
        if (!(sd > 1.0e-8) || !isfinite(sd)) *bad = 1;            // inference.py:564 (cannot happen for Gaussian z, n >= 2)
        stats[row] = make_double2(mean, sd);
    }
}

// out = template * (raw - mean) / sd   (in place over raw)
__global__ void __launch_bounds__(256) k_wild_apply(const double *__restrict__ T, double *__restrict__ W, long long n,
                                                    const double2 *__restrict__ stats)
{
    const long long row = blockIdx.y;
    const double2 ms = stats[row];
    const double rsd = 1.0 / ms.y;
    const double *t = T + row * n;
    double *w = W + row * n;
    for (long long j = (long long)blockIdx.x * blockDim.x + threadIdx.x; j < n; j += (long long)gridDim.x * blockDim.x)
        w[j] = t[j] * score::div_rcp(w[j] - ms.x, ms.y, rsd);
}

// ------------------------------------------------------------------ reductions over a score track
// sums of  (s-c)+ , (s-c)+/soft , [(s-c)+ > 0] , [s > thr] , [s < c] , s is finite ;  fixed order: per-CTA partials, one CTA
__global__ void __launch_bounds__(RED_THREADS) k_track_partial(const double *__restrict__ s, long long n, double c, double soft,
                                                               double thr, double *__restrict__ part /* [grid][6] */)
{
    double a[6] = {0, 0, 0, 0, 0, 0};
    for (long long j = (long long)blockIdx.x * RED_THREADS + threadIdx.x; j < n; j += (long long)gridDim.x * RED_THREADS) {
        const double v = s[j];
        const double pos = fmax(v - c, 0.0);
        a[0] += pos; a[1] += pos / soft; a[2] += (pos > 0.0) ? 1.0 : 0.0; a[3] += (v > thr) ? 1.0 : 0.0;
        a[4] += (v < c) ? 1.0 : 0.0; a[5] += isfinite(v) ? 0.0 : 1.0;
    }
    __shared__ double sh[6][RED_THREADS / 32];
#pragma unroll
    for (int q = 0; q < 6; ++q) {
        double v = a[q];
#pragma unroll
        for (int d = 16; d > 0; d >>= 1) v += __shfl_down_sync(0xffffffffu, v, d);
        if ((threadIdx.x & 31) == 0) sh[q][threadIdx.x >> 5] = v;
    }
    __syncthreads();
    if (threadIdx.x < 6) {
        double v = 0.0;
        for (int w = 0; w < RED_THREADS / 32; ++w) v += sh[threadIdx.x][w];
        part[(long long)blockIdx.x * 6 + threadIdx.x] = v;
    }
}

__global__ void __launch_bounds__(256) k_partial_final(const double *__restrict__ part, int blocks, int width, double *out)
{
    __shared__ double sh[256];
    for (int q = 0; q < width; ++q) {
        double v = 0.0;
        for (int b = threadIdx.x; b < blocks; b += 256) v += part[(long long)b * width + q];
        sh[threadIdx.x] = v;
        __syncthreads();
        for (int d = 128; d > 0; d >>= 1) { if (threadIdx.x < d) sh[threadIdx.x] += sh[threadIdx.x + d]; __syncthreads(); }
        if (threadIdx.x == 0) out[q] = sh[0];
        __syncthreads();
    }
}

// sum and max of max(mean, 0)
__global__ void __launch_bounds__(RED_THREADS) k_consensus_partial(const double *__restrict__ mean, long long n, double *part)
{
    double a = 0.0, mx = 0.0;
    for (long long j = (long long)blockIdx.x * RED_THREADS + threadIdx.x; j < n; j += (long long)gridDim.x * RED_THREADS) {
        const double v = fmax(mean[j], 0.0);
        a += v; mx = fmax(mx, v);
    }
    __shared__ double sh[2][RED_THREADS / 32];
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) { a += __shfl_down_sync(0xffffffffu, a, d); mx = fmax(mx, __shfl_down_sync(0xffffffffu, mx, d)); }
    if ((threadIdx.x & 31) == 0) { sh[0][threadIdx.x >> 5] = a; sh[1][threadIdx.x >> 5] = mx; }
    __syncthreads();
    if (threadIdx.x == 0) {
        double s = 0.0, m2 = 0.0;
        for (int w = 0; w < RED_THREADS / 32; ++w) { s += sh[0][w]; m2 = fmax(m2, sh[1][w]); }
        part[(long long)blockIdx.x * 2] = s; part[(long long)blockIdx.x * 2 + 1] = m2;
    }
}
__global__ void k_consensus_final(const double *part, int blocks, double *out)
{
    if (threadIdx.x == 0 && blockIdx.x == 0) {
        double s = 0.0, mx = 0.0;
        for (int b = 0; b < blocks; ++b) { s += part[2 * b]; mx = fmax(mx, part[2 * b + 1]); }
        out[0] = s; out[1] = mx;
    }
}

// ------------------------------------------------------------------ order statistics of a sorted track
// out[0] = median, out[1] = 1.4826 * MAD of the mirrored non-positive residuals (floored), out[2] = their count
// (inference.py:768-783).  With r = s - center sorted ascending, the k residuals <= 0 give magnitudes
// mag_j = center - s[k-1-j] (ascending in j); the mirrored set {-mag, +mag} has median exactly 0 and its absolute
// values are each magnitude twice, so the MAD is (mag[(k-1)/2] + mag[k/2]) / 2.
__global__ void k_center_scale(const double *__restrict__ sorted, long long n, double *out)
{
    if (threadIdx.x || blockIdx.x) return;
    const double center = (n & 1) ? sorted[n / 2] : 0.5 * (sorted[n / 2 - 1] + sorted[n / 2]);
    long long lo = 0, hi = n;                                  // k = #(s <= center)
    while (lo < hi) { const long long mid = (lo + hi) >> 1; if (sorted[mid] <= center) lo = mid + 1; else hi = mid; }
    const long long k = lo;
    double mad = 0.0;
    if (k > 0) {
        const double m_lo = -(sorted[k - 1 - (k - 1) / 2] - center), m_hi = -(sorted[k - 1 - k / 2] - center);
        mad = 0.5 * (m_lo + m_hi);
    }
    out[0] = center;
    out[1] = fmax(mad * 1.4826, 1.0e-6);
    out[2] = (double)k;
}

// median and count of the strictly positive entries of a sorted track (rocco.py:762-769)
__global__ void k_positive_median(const double *__restrict__ sorted, long long n, double *out)
{
    if (threadIdx.x || blockIdx.x) return;
    long long lo = 0, hi = n;                                  // first index with s > 0
    while (lo < hi) { const long long mid = (lo + hi) >> 1; if (sorted[mid] > 0.0) hi = mid; else lo = mid + 1; }
    const long long p = n - lo;
    double med = 1.0;
    if (p > 0) med = (p & 1) ? sorted[lo + p / 2] : 0.5 * (sorted[lo + p / 2 - 1] + sorted[lo + p / 2]);
    out[0] = med;
    out[1] = (double)p;
}

// ------------------------------------------------------------------ autocovariances by direct lag products
// v_j = transform ? max(s_j - c, 0) / soft : s_j ;  x = v - mean ;  part[tile][l] = sum_{j in tile, j + l < n} x_j x_{j+l}
__global__ void __launch_bounds__(AC_THREADS) k_autocov_partial(const double *__restrict__ s, long long n, int transform, double c,
                                                                double soft, double mean, int L, double *__restrict__ part)
{
    extern __shared__ double s_ac[];                           // AC_T + L
    const long long j0 = (long long)blockIdx.x * AC_T;
    const int span = (int)min((long long)(AC_T + L), n - j0);
    const int own = (int)min((long long)AC_T, n - j0);
    for (int e = threadIdx.x; e < AC_T + L; e += AC_THREADS) {
        double v = 0.0;
        if (e < span) {
            v = s[j0 + e];
            if (transform) v = fmax(v - c, 0.0) / soft;
            v -= mean;
        }
        s_ac[e] = v;
    }
    __syncthreads();
    for (int l = threadIdx.x; l <= L; l += AC_THREADS) {
        double a0 = 0.0, a1 = 0.0, a2 = 0.0, a3 = 0.0;
        int j = 0;
        for (; j + 4 <= own; j += 4) {
            a0 = fma(s_ac[j], s_ac[j + l], a0); a1 = fma(s_ac[j + 1], s_ac[j + 1 + l], a1);
            a2 = fma(s_ac[j + 2], s_ac[j + 2 + l], a2); a3 = fma(s_ac[j + 3], s_ac[j + 3 + l], a3);
        }
        for (; j < own; ++j) a0 = fma(s_ac[j], s_ac[j + l], a0);
        part[(long long)blockIdx.x * (L + 1) + l] = (a0 + a1) + (a2 + a3);     // entries past the end are zero-padded
    }
}

__global__ void __launch_bounds__(256) k_autocov_final(const double *__restrict__ part, int tiles, int L, long long n, double *acov)
{
    const int l = blockIdx.x;
    __shared__ double sh[256];
    double v = 0.0;
    for (int t = threadIdx.x; t < tiles; t += 256) v += part[(long long)t * (L + 1) + l];
    sh[threadIdx.x] = v;
    __syncthreads();
    for (int d = 128; d > 0; d >>= 1) { if (threadIdx.x < d) sh[threadIdx.x] += sh[threadIdx.x + d]; __syncthreads(); }
    if (threadIdx.x == 0) acov[l] = sh[0] / (double)(n - l);
}

// ------------------------------------------------------------------ sample sharding: status slots of a reduce
// After the 2n column sums of a sharded reduce: slot k counts the ranks that failed with status -(k + 1) (ST_NOMEM,
// ST_INVALID, ST_CUDA, ST_NONFINITE).  Summed, the slots are the same on every rank, and so is the status they return.
constexpr int NSTATUS = 4;

__global__ void k_shard_status(double *slots, int local_status, const int *bad)
{
    const int k = threadIdx.x;
    if (k >= NSTATUS) return;
    const int cls = (local_status >= -NSTATUS && local_status < 0) ? -local_status - 1 : (local_status ? -ST_CUDA - 1 : -1);
    double v = (k == cls) ? 1.0 : 0.0;
    if (k == -ST_NONFINITE - 1 && bad && *bad) v += 1.0;        // degenerate multiplier row of this rank
    slots[k] = v;
}

// ------------------------------------------------------------------ host side
static size_t sort_track_bytes(long long n)
{
    size_t bytes = 0;
    cub::DeviceRadixSort::SortKeys(nullptr, bytes, (const double *)nullptr, (double *)nullptr, (int)n, 0, 64);
    return bytes;
}

// `tmp` holds sort_track_bytes(n)
static int sort_track(char *tmp, const double *d_in, double *d_sorted, long long n, cudaStream_t st)
{
    size_t bytes = sort_track_bytes(n);
    RB_CUDA(cub::DeviceRadixSort::SortKeys(tmp, bytes, d_in, d_sorted, (int)n, 0, 64, st));
    count_launch(4);
    return 0;
}

static int track_sums(const double *d_s, long long n, double c, double soft, double thr, double *d_part, double *d_out6,
                      double *h6, cudaStream_t st)
{
    const int blocks = (int)std::min<long long>(RED_BLOCKS, (n + RED_THREADS - 1) / RED_THREADS);
    k_track_partial<<<blocks, RED_THREADS, 0, st>>>(d_s, n, c, soft, thr, d_part);
    RB_LAUNCH_CHECK();
    k_partial_final<<<1, 256, 0, st>>>(d_part, blocks, 6, d_out6);
    RB_LAUNCH_CHECK();
    RB_CUDA(cudaMemcpyAsync(h6, d_out6, 6 * sizeof(double), cudaMemcpyDeviceToHost, st));
    RB_CUDA(cudaStreamSynchronize(st));
    return 0;
}

static double bartlett_taps(int b, std::vector<double> &taps)          // returns the slope h: taps[k] = h (b + 1 - |k - b|)
{
    // inference.py:533-541, same operation order as NumPy: maximum(1 - |k| / (b + 1), 0) / sqrt(sum of squares)
    taps.resize((size_t)(2 * b + 1));
    for (int k = -b; k <= b; ++k) taps[(size_t)(k + b)] = std::max(1.0 - std::fabs((double)k) / (double)(b + 1), 0.0);
    std::vector<double> sq(taps.size());
    for (size_t i = 0; i < taps.size(); ++i) sq[i] = taps[i] * taps[i];
    const double nrm = std::sqrt(numpy_sum_f64(sq.data(), sq.size()));
    for (double &t : taps) t /= nrm;
    return 1.0 / ((double)(b + 1) * nrm);
}

int resolve_bandwidth(long long n, int hint)
{
    if (n <= 1) return 1;
    long long want = hint > 0 ? hint : (long long)std::nearbyint(std::pow((double)n, 1.0 / 3.0));
    return (int)std::min<long long>(n - 1, std::max<long long>(8, want));
}

int resolve_ess_max_lag(long long n, int hint)
{
    const long long n_ = std::max<long long>(1, n);
    const long long base = hint > 0 ? std::max<long long>(1, std::min<long long>(n_, hint)) : std::min<long long>(n_, 101);
    return (int)std::min<long long>(n_ - 1, std::max<long long>(16, 4 * base));
}

struct Welford {
    int n = 0; double mean = 0.0, m2 = 0.0;
    void add(double x) { ++n; const double d = x - mean; mean += d / (double)n; m2 += d * (x - mean); }
    double var() const { return std::max(m2 / (double)std::max(n - 1, 1), 0.0); }
    double sd() const { return std::sqrt(var()); }
    double stderr_() const { return std::sqrt(var() / (double)std::max(n, 1)); }
};

// scratch of wild_multiply: per-(row, tile) partial moments, then per-row (mean, sd)
struct WildScratch {
    double2 *part = nullptr, *stats = nullptr;
    int alloc(Arena &ar, long long m, long long n)
    {
        RB_TRY(ar.alloc(&part, (size_t)m * (size_t)((n + FIR_T - 1) / FIR_T)));
        return ar.alloc(&stats, (size_t)m);
    }
};

// NumPy streams of an estimator call: draw d is default_rng(seed + 104729 (d + 1)); global sample i takes its normals
// [i L, (i + 1) L), L = n + 2 bandwidth.  Rows are generated `rows` at a time into `buf` (at most 256 MB), each group
// continuing the stream where the previous one stopped.
struct NumpyField {
    static constexpr long long MAX_BUF = 32LL << 20;      // doubles
    double *buf = nullptr;
    long long rows = 0;
    npz::Scratch sc;
    int alloc(Arena &ar, long long m, long long L, long long sample_offset)
    {
        rows = std::max(1LL, std::min(m, MAX_BUF / L));
        RB_TRY(ar.alloc(&buf, (size_t)(rows * L)));
        return sc.alloc(ar, std::max(rows, sample_offset) * L);
    }
};

// one multiplier field applied to the template:  d_out = template x W   (inference.py:656-662); row r draws the stream of
// sample sample_offset + r (Philox; with `np` the NumPy stream of that draw, unless d_innov is given)
static int wild_multiply(const WildScratch &ws, const double *d_template, long long m, long long n, int bandwidth, const double *d_taps,
                         double h, unsigned long long seed, unsigned draw, unsigned sample_offset, const double *d_innov, double *d_out,
                         int *d_bad, cudaStream_t st, NumpyField *np = nullptr)
{
    if (n == 1) {                                         // weights are exactly one (inference.py:556-557)
        RB_CUDA(cudaMemcpyAsync(d_out, d_template, sizeof(double) * (size_t)m, cudaMemcpyDeviceToDevice, st));
        return 0;
    }
    const int K = 2 * bandwidth + 1;
    const int tiles = (int)((n + FIR_T - 1) / FIR_T);
    double2 *d_part = ws.part, *d_stats = ws.stats;
    const size_t smem = sizeof(double) * ((size_t)padpos(FIR_T + K + 8) + 8 + (size_t)K);
    static bool attr_dev[64] = {false};
    int dev = 0;
    cudaGetDevice(&dev);
    if (!attr_dev[dev & 63]) {
        RB_CUDA(cudaFuncSetAttribute(k_wild_fir, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                     (int)(sizeof(double) * ((size_t)padpos(FIR_T + 2 * MAX_BANDWIDTH + 1 + 8) + 8 + 2 * MAX_BANDWIDTH + 1))));
        attr_dev[dev & 63] = true;
    }
    const uint2 key = make_uint2((unsigned)seed, (unsigned)(seed >> 32));
    if (np && !d_innov) {
        const long long L = n + K - 1;
        npz::Cursor cur = npz::seed_cursor((npz::u128)seed + (npz::u128)104729 * ((npz::u128)draw + 1));
        for (long long r0 = 0; r0 < m; r0 += np->rows) {
            const long long r1 = std::min(m, r0 + np->rows);
            RB_TRY(npz::generate(cur, ((long long)sample_offset + r0) * L, ((long long)sample_offset + r1) * L, np->buf, nullptr, np->sc, st));
            RB_PROF("k_wild_fir", st, (double)(r1 - r0) * n * 8.0);
            k_wild_fir<<<dim3((unsigned)tiles, (unsigned)(r1 - r0)), FIR_THREADS, smem, st>>>(np->buf, L, key, draw, sample_offset + (unsigned)r0,
                                                                                             n, K, d_taps, h, d_out + r0 * n,
                                                                                             d_part + r0 * tiles, tiles);
            RB_LAUNCH_CHECK();
        }
    } else {
        RB_PROF("k_wild_fir", st, (double)m * n * 8.0);
        k_wild_fir<<<dim3((unsigned)tiles, (unsigned)m), FIR_THREADS, smem, st>>>(d_innov, n + K - 1, key, draw, sample_offset, n, K,
                                                                                  d_taps, h, d_out, d_part, tiles);
        RB_LAUNCH_CHECK();
    }
    k_row_moments<<<(unsigned)m, 256, 0, st>>>(d_part, tiles, n, d_stats, d_bad);
    RB_LAUNCH_CHECK();
    {
        RB_PROF("k_wild_apply", st, (double)m * n * 24.0);
        const unsigned gx = (unsigned)std::min<long long>((n + 256 * 8 - 1) / (256 * 8), 65535);
        k_wild_apply<<<dim3(gx, (unsigned)m), 256, 0, st>>>(d_template, d_out, n, d_stats);
        RB_LAUNCH_CHECK();
    }
    return 0;
}

static int autocov(Arena &ar, const double *d_s, long long n, int transform, double c, double soft, double mean, int L,
                   double *h_acov, cudaStream_t st)
{
    const int tiles = (int)((n + AC_T - 1) / AC_T);
    double *d_part = nullptr, *d_acov = nullptr;
    RB_TRY(ar.alloc(&d_part, (size_t)tiles * (L + 1)));
    RB_TRY(ar.alloc(&d_acov, (size_t)L + 1));
    static bool attr_dev[64] = {false};
    int dev = 0;
    cudaGetDevice(&dev);
    if (!attr_dev[dev & 63]) {
        RB_CUDA(cudaFuncSetAttribute(k_autocov_partial, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                     (int)(sizeof(double) * (AC_T + AC_MAXLAG))));
        attr_dev[dev & 63] = true;
    }
    k_autocov_partial<<<tiles, AC_THREADS, sizeof(double) * (size_t)(AC_T + L), st>>>(d_s, n, transform, c, soft, mean, L, d_part);
    RB_LAUNCH_CHECK();
    k_autocov_final<<<L + 1, 256, 0, st>>>(d_part, tiles, L, n, d_acov);
    RB_LAUNCH_CHECK();
    RB_CUDA(cudaMemcpyAsync(h_acov, d_acov, sizeof(double) * (size_t)(L + 1), cudaMemcpyDeviceToHost, st));
    RB_CUDA(cudaStreamSynchronize(st));
    return 0;
}

// Geyer's initial positive sequence on the autocorrelations (inference.py:481-501)
static void geyer(const double *acov, long long n, int L, double *n_eff, double *tau_out, int *lags_used)
{
    double tau = 1.0;
    int used = 0;
    for (int k = 0; k < L; k += 2) {
        auto rho = [&](int q) { return std::min(1.0, std::max(-1.0, acov[q + 1] / acov[0])); };
        const double pair = rho(k) + ((k + 1 < L) ? rho(k + 1) : 0.0);
        if (!std::isfinite(pair) || pair <= 0.0) break;
        tau += 2.0 * pair;
        used = std::min(L, k + 2);
    }
    *tau_out = tau;
    *lags_used = used;
    *n_eff = std::min((double)n, std::max(1.0, (double)n / std::max(tau, 1.0)));
}

static int effective_sample_size(Arena &ar, const double *d_s, long long n, int transform, double c, double soft, double mean,
                                 int max_lag, double *n_eff, double *tau, int *used, cudaStream_t st)
{
    *n_eff = (double)std::max<long long>(1, n); *tau = 1.0; *used = 0;
    if (n < 4) return 0;
    const int L = (int)std::min<long long>(std::max(2, max_lag), n - 1);
    if (L > AC_MAXLAG) { set_error("autocovariance lag cap %d exceeds %d", L, AC_MAXLAG); return ST_INVALID; }
    std::vector<double> acov((size_t)L + 1);
    RB_TRY(autocov(ar, d_s, n, transform, c, soft, mean, L, acov.data(), st));
    *n_eff = (double)n;
    if (!std::isfinite(acov[0]) || acov[0] <= 1.0e-12) return 0;
    geyer(acov.data(), n, L, n_eff, tau, used);
    return 0;
}

// Sample sharding of one estimator call.  reduce == nullptr: one rank holds every sample and each step runs as written.
struct Shard {
    rocco_b200_allreduce_fn reduce = nullptr;
    void *user = nullptr;
    long long m_total = 0;
    double *d_red = nullptr;      // [2n column sums][NSTATUS status slots], the buffer every pass reduces
    int *d_fin_bad = nullptr;     // non-finite flag of the finalisation
    int failed = 0;               // first rank-local failure; the rank's local work stops until the next reduce reports it

    // A rank-local step.  Unsharded its failure is returned at once; sharded it is kept for the next reduce (all ranks must
    // get there) and 0 is returned.
    int local(int status)
    {
        if (status == 0 || !reduce) return status;
        if (!failed) failed = status;
        return 0;
    }
};

// One scoring pass over this rank's rows -> d_scores (and d_mean when not null).  Unsharded: the centred-WLS chain.  Sharded:
// the per-row stages and the partial column sums (skipped after a local failure), the status slots, the reduce, and the
// finalisation of the summed sums; every rank returns the same status.
static int score_pass(Shard &S, const double *d_rows, long long m, long long n, const rocco_b200_score_params &prm, double *d_scores,
                      double *d_mean, const int *d_bad, cudaStream_t st)
{
    rocco_b200_score_outputs so{};
    so.scores = d_scores; so.mean = d_mean;
    if (!S.reduce) return score::centered_wls(d_rows, m, n, prm, &so, st);
    if (!S.failed) {
        rocco_b200_score_outputs none{};
        S.local(score::centered_wls(d_rows, m, n, prm, &none, st, S.d_red));
    }
    k_shard_status<<<1, 32, 0, st>>>(S.d_red + 2 * n, S.failed, d_bad);
    count_launch();
    S.local(cudaGetLastError() == cudaSuccess ? 0 : ST_CUDA);
    if (S.reduce(S.d_red, (size_t)(2 * n + NSTATUS), (void *)st, S.user) != 0) {
        set_error("sample-sharded budget null: the all-reduce callback failed");
        return ST_CUDA;
    }
    RB_TRY(score::finalize_acc(S.d_red, n, false, S.m_total, prm, &so, S.d_fin_bad, st));
    double slots[NSTATUS];
    int flags[2] = {0, 0};
    RB_CUDA(cudaMemcpyAsync(slots, S.d_red + 2 * n, sizeof(slots), cudaMemcpyDeviceToHost, st));
    RB_CUDA(cudaMemcpyAsync(&flags[0], S.d_fin_bad, sizeof(int), cudaMemcpyDeviceToHost, st));
    if (d_bad) RB_CUDA(cudaMemcpyAsync(&flags[1], d_bad, sizeof(int), cudaMemcpyDeviceToHost, st));
    RB_CUDA(cudaStreamSynchronize(st));
    for (int k = 0; k < NSTATUS; ++k) {
        if (!(slots[k] > 0.0)) continue;
        if (flags[1]) set_error("degenerate multiplier field");
        else if (!S.failed) set_error("sample-sharded budget null: another rank failed with status %d", -(k + 1));
        return -(k + 1);
    }
    return flags[0] ? ST_NONFINITE : 0;
}

static int budget_core(const double *d_centered, long long m, long long n, const double *d_observed, const rocco_b200_budget_params &P,
                       Shard &S, rocco_b200_budget_result *R, cudaStream_t st)
{
    if (!d_centered || !R || m <= 0 || n <= 0) return ST_INVALID;
    RB_TRY(ensure_device());
    memset(R, 0, sizeof(*R));
    Arena ar(st);
    const int bandwidth = resolve_bandwidth(n, P.dependence_lag_hint);
    if (bandwidth > MAX_BANDWIDTH) { set_error("bootstrap bandwidth %d exceeds %d", bandwidth, MAX_BANDWIDTH); return ST_INVALID; }
    double *d_fit = nullptr, *d_mean = nullptr, *d_tmpl = nullptr, *d_boot = nullptr, *d_ref = nullptr, *d_sorted = nullptr;
    double *d_part = nullptr, *d_small = nullptr, *d_taps = nullptr;
    char *d_sort_tmp = nullptr;
    int *d_bad = nullptr;
    WildScratch wild;
    NumpyField numpy_field;
    const bool numpy_streams = P.random_streams == 1 && !P.d_innovations && n > 1;
    if (S.reduce) {
        // the buffers every pass needs to take part in a reduce (a failure here cannot be reported to the other ranks)
        RB_TRY(ar.alloc(&S.d_red, (size_t)(2 * n + NSTATUS)));
        RB_TRY(ar.alloc(&S.d_fin_bad, 1));
        RB_CUDA(cudaMemsetAsync(S.d_fin_bad, 0, sizeof(int), st));
    }
    std::vector<double> taps;
    const double tap_step = bartlett_taps(bandwidth, taps);
    // everything the passes and the draw loop need, before the first reduce
    auto setup = [&]() -> int {
        RB_TRY(ar.alloc(&d_bad, 1));
        RB_CUDA(cudaMemsetAsync(d_bad, 0, sizeof(int), st));
        RB_TRY(ar.alloc(&d_fit, (size_t)n));
        RB_TRY(ar.alloc(&d_mean, (size_t)n));
        RB_TRY(ar.alloc(&d_ref, (size_t)n));
        RB_TRY(ar.alloc(&d_sorted, (size_t)n));
        RB_TRY(ar.alloc(&d_tmpl, (size_t)m * n));
        RB_TRY(ar.alloc(&d_boot, (size_t)m * n));
        RB_TRY(ar.alloc(&d_part, (size_t)RED_BLOCKS * 6));
        RB_TRY(ar.alloc(&d_small, 16));
        RB_TRY(ar.alloc(&d_sort_tmp, sort_track_bytes(n)));
        RB_TRY(wild.alloc(ar, m, n));
        if (numpy_streams) RB_TRY(numpy_field.alloc(ar, m, n + 2LL * bandwidth, P.sample_offset));
        RB_TRY(ar.alloc(&d_taps, taps.size()));
        RB_CUDA(cudaMemcpyAsync(d_taps, taps.data(), sizeof(double) * taps.size(), cudaMemcpyHostToDevice, st));
        return 0;
    };
    RB_TRY(S.local(setup()));

    // ---- fit, template, fitted-null score field
    RB_TRY(score_pass(S, d_centered, m, n, P.score, d_fit, d_mean, d_bad, st));
    if (!S.failed) {
        const long long total = m * n;
        const unsigned grid = (unsigned)std::min<long long>((total + 255) / 256, 148LL * 32);
        k_template<<<grid, 256, 0, st>>>(d_centered, d_mean, m, n, d_tmpl);
        count_launch();
        RB_TRY(S.local(cudaGetLastError() == cudaSuccess ? 0 : ST_CUDA));
    }
    double h[8];
    {
        const int blocks = (int)std::min<long long>(RED_BLOCKS, (n + RED_THREADS - 1) / RED_THREADS);
        k_consensus_partial<<<blocks, RED_THREADS, 0, st>>>(d_mean, n, d_part);
        RB_LAUNCH_CHECK();
        k_consensus_final<<<1, 32, 0, st>>>(d_part, blocks, d_small);
        RB_LAUNCH_CHECK();
        RB_CUDA(cudaMemcpyAsync(h, d_small, 2 * sizeof(double), cudaMemcpyDeviceToHost, st));
        RB_CUDA(cudaStreamSynchronize(st));
        R->null_reference_mean_positive_consensus = h[0] / (double)n;
        R->null_reference_max_positive_consensus = h[1];
    }
    RB_TRY(score_pass(S, d_tmpl, m, n, P.score, d_ref, nullptr, d_bad, st));
    RB_TRY(sort_track(d_sort_tmp, d_ref, d_sorted, n, st));
    k_center_scale<<<1, 32, 0, st>>>(d_sorted, n, d_small);
    RB_LAUNCH_CHECK();
    RB_CUDA(cudaMemcpyAsync(h, d_small, 3 * sizeof(double), cudaMemcpyDeviceToHost, st));
    RB_CUDA(cudaStreamSynchronize(st));
    const double center = h[0], scale = h[1];
    if (!std::isfinite(center) || !std::isfinite(scale)) return ST_NONFINITE;
    const double soft = std::max(scale, 1.0e-6), threshold = center + 2.0 * scale;
    R->null_center = center; R->null_scale = scale; R->null_threshold = threshold;
    R->negative_support_size = (long long)h[2];
    R->negative_fraction = h[2] / (double)std::max<long long>(n, 1);
    R->wild_bandwidth = bandwidth;

    // ---- draws (inference.py:800-880): Welford moments of the four per-draw means, stop once the soft-count mean is stable
    const int draws = std::max(1, P.num_null_draws);
    const int min_draws = std::min(draws, std::max(4, P.min_null_draws > 0 ? P.min_null_draws : 8));
    Welford acc[4];
    const size_t innov_per_draw = (size_t)m * (size_t)(n + 2 * bandwidth);
    for (int d = 0; d < draws; ++d) {
        const double *innov = P.d_innovations ? P.d_innovations + (size_t)d * innov_per_draw : nullptr;
        if (!S.failed)
            RB_TRY(S.local(wild_multiply(wild, d_tmpl, m, n, bandwidth, d_taps, tap_step, P.random_seed, (unsigned)d,
                                         (unsigned)P.sample_offset, innov, d_boot, d_bad, st,
                                         numpy_streams ? &numpy_field : nullptr)));
        // the reference field is no longer needed: reuse its buffer
        RB_TRY(score_pass(S, d_boot, m, n, P.score, d_ref, nullptr, d_bad, st));
        RB_TRY(track_sums(d_ref, n, center, soft, threshold, d_part, d_small, h, st));
        if (h[5] != 0.0) return ST_NONFINITE;
        for (int q = 0; q < 4; ++q) acc[q].add(h[q] / (double)n);
        if (acc[1].n >= std::max(2, min_draws)) {
            const double target = std::max(P.stability_abs_tol, P.stability_rel_tol * std::max(std::fabs(acc[1].mean), 1.0e-6));
            if (acc[1].stderr_() <= target) break;
        }
    }
    int bad = 0;
    RB_CUDA(cudaMemcpyAsync(&bad, d_bad, sizeof(int), cudaMemcpyDeviceToHost, st));
    RB_CUDA(cudaStreamSynchronize(st));
    if (bad) { set_error("degenerate multiplier field"); return ST_NONFINITE; }
    R->num_null_draws = acc[0].n; R->max_null_draws = draws; R->adaptive_stop = acc[0].n < draws;
    R->null_positive_mass = acc[0].mean; R->null_positive_units = acc[1].mean; R->null_positive_fraction = acc[2].mean;
    R->null_positive_units_sd = acc[1].sd(); R->null_positive_units_stderr = acc[1].stderr_();
    R->null_tail_occupancy = acc[3].mean; R->null_tail_occupancy_sd = acc[3].sd(); R->null_tail_occupancy_stderr = acc[3].stderr_();

    // ---- observed side (inference.py:1063-1100)
    const double *d_obs = d_observed ? d_observed : d_fit;
    RB_TRY(track_sums(d_obs, n, center, soft, threshold, d_part, d_small, h, st));
    if (h[5] != 0.0) return ST_NONFINITE;
    R->observed_excess_mass = h[0] / (double)n; R->observed_excess_units = h[1] / (double)n;
    R->observed_positive_fraction = h[2] / (double)n; R->observed_tail_occupancy = h[3] / (double)n;
    R->observed_negative_fraction = h[4] / (double)n;
    R->ess_max_lag = resolve_ess_max_lag(n, P.dependence_lag_hint);
    RB_TRY(effective_sample_size(ar, d_obs, n, 1, center, soft, R->observed_excess_units, R->ess_max_lag, &R->effective_total_count,
                                 &R->autocorrelation_time, &R->ess_lags_used, st));
    R->nonnull_fraction = std::min(1.0, std::max(0.0, R->observed_tail_occupancy - R->null_tail_occupancy));
    if (!std::isfinite(R->nonnull_fraction) || !std::isfinite(R->effective_total_count) || !std::isfinite(R->autocorrelation_time))
        return ST_NONFINITE;
    R->effective_count = R->nonnull_fraction * R->effective_total_count;
    R->num_loci = n;
    // ---- automatic gamma inputs (rocco.py:762-769)
    RB_TRY(sort_track(d_sort_tmp, d_obs, d_sorted, n, st));
    k_positive_median<<<1, 32, 0, st>>>(d_sorted, n, d_small);
    RB_LAUNCH_CHECK();
    RB_CUDA(cudaMemcpyAsync(h, d_small, 2 * sizeof(double), cudaMemcpyDeviceToHost, st));
    RB_CUDA(cudaStreamSynchronize(st));
    R->positive_score_median = h[0];
    R->positive_score_count = (long long)h[1];
    return 0;
}

}  // namespace budget
}  // namespace rb

// ==================================================================================== C ABI
using namespace rb;
#define RB_API __attribute__((visibility("default")))

extern "C" {

RB_API void rocco_b200_default_budget_params(rocco_b200_budget_params *p)
{
    if (!p) return;
    memset(p, 0, sizeof(*p));
    rocco_b200_default_score_params(&p->score);
    p->dependence_lag_hint = 0;
    p->num_null_draws = 25;
    p->min_null_draws = 0;
    p->stability_abs_tol = 5.0e-3;
    p->stability_rel_tol = 5.0e-2;
    p->random_seed = 0;
    p->d_innovations = nullptr;
    p->random_streams = 0;
}

RB_API int rocco_b200_budget_bandwidth(size_t n, int dependence_lag_hint) { return budget::resolve_bandwidth((long long)n, dependence_lag_hint); }
RB_API int rocco_b200_budget_ess_max_lag(size_t n, int dependence_lag_hint) { return budget::resolve_ess_max_lag((long long)n, dependence_lag_hint); }

RB_API int rocco_b200_budget_nonnull_fraction_dev(const double *d_centered, size_t m, size_t n, const double *d_observed_scores,
                                                  const rocco_b200_budget_params *params, rocco_b200_budget_result *result,
                                                  void *cuda_stream)
{
    rocco_b200_budget_params P;
    if (params) P = *params; else rocco_b200_default_budget_params(&P);
    if (P.sample_offset < 0 || P.random_streams < 0 || P.random_streams > 1) return ST_INVALID;
    budget::Shard whole;
    return budget::budget_core(d_centered, (long long)m, (long long)n, d_observed_scores, P, whole, result, (cudaStream_t)cuda_stream);
}

RB_API int rocco_b200_budget_nonnull_fraction_sharded_dev(const double *d_centered_local, size_t m_local, size_t n, size_t m_total,
                                                          const double *d_observed_scores, const rocco_b200_budget_params *params,
                                                          rocco_b200_allreduce_fn allreduce, void *user, rocco_b200_budget_result *result,
                                                          void *cuda_stream)
{
    rocco_b200_budget_params P;
    if (params) P = *params; else rocco_b200_default_budget_params(&P);
    if (m_local == 0 || P.sample_offset < 0 || (size_t)P.sample_offset + m_local > m_total) return ST_INVALID;
    if (P.random_streams < 0 || P.random_streams > 1) return ST_INVALID;
    if (!allreduce && m_local != m_total) return ST_INVALID;
    budget::Shard shard;
    shard.reduce = allreduce;
    shard.user = user;
    shard.m_total = (long long)m_total;
    return budget::budget_core(d_centered_local, (long long)m_local, (long long)n, d_observed_scores, P, shard, result,
                               (cudaStream_t)cuda_stream);
}

// One bootstrap draw's input (inference.py:653-662): d_out[i][j] = d_template[i][j] * W_ij with W the unit-variance
// Bartlett-smoothed multiplier field of (random_seed, draw) -- or of the supplied innovations [m][n + 2*bandwidth].
RB_API int rocco_b200_wild_multiply_dev(const double *d_template, size_t m, size_t n, int bandwidth, unsigned long long random_seed,
                                        unsigned draw_index, const double *d_innovations, double *d_out, void *cuda_stream)
{
    if (!d_template || !d_out || m == 0 || n == 0 || bandwidth < 1 || bandwidth > budget::MAX_BANDWIDTH) return ST_INVALID;
    RB_TRY(ensure_device());
    cudaStream_t st = (cudaStream_t)cuda_stream;
    Arena ar(st);
    std::vector<double> taps;
    const double tap_step = budget::bartlett_taps(bandwidth, taps);
    double *d_taps = nullptr;
    int *d_bad = nullptr;
    budget::WildScratch ws;
    RB_TRY(ws.alloc(ar, (long long)m, (long long)n));
    RB_TRY(ar.alloc(&d_taps, taps.size()));
    RB_TRY(ar.alloc(&d_bad, 1));
    RB_CUDA(cudaMemsetAsync(d_bad, 0, sizeof(int), st));
    RB_CUDA(cudaMemcpyAsync(d_taps, taps.data(), sizeof(double) * taps.size(), cudaMemcpyHostToDevice, st));
    RB_TRY(budget::wild_multiply(ws, d_template, (long long)m, (long long)n, bandwidth, d_taps, tap_step, random_seed, draw_index, 0,
                                 d_innovations, d_out, d_bad, st));
    int bad = 0;
    RB_CUDA(cudaMemcpyAsync(&bad, d_bad, sizeof(int), cudaMemcpyDeviceToHost, st));
    RB_CUDA(cudaStreamSynchronize(st));                   // also keeps `taps` alive until the copy has been consumed
    return bad ? ST_NONFINITE : 0;
}

// Host-pointer form: centered matrix (and optional observed scores / innovations) live in host memory.
RB_API int rocco_budget_nonnull_fraction_f64(const double *centered, size_t m, size_t n, const double *observed_scores,
                                             const rocco_b200_budget_params *params, const double *innovations,
                                             rocco_b200_budget_result *result)
{
    if (!centered || !result || m == 0 || n == 0) return ST_INVALID;
    RB_TRY(ensure_device());
    rocco_b200_budget_params P;
    if (params) P = *params; else rocco_b200_default_budget_params(&P);
    HostScope lease;
    cudaStream_t st = lease.stream();
    Arena ar(st);
    double *d_c = nullptr, *d_o = nullptr, *d_i = nullptr;
    RB_TRY(ar.alloc(&d_c, m * n));
    RB_CUDA(cudaMemcpyAsync(d_c, centered, sizeof(double) * m * n, cudaMemcpyHostToDevice, st));
    if (observed_scores) {
        RB_TRY(ar.alloc(&d_o, n));
        RB_CUDA(cudaMemcpyAsync(d_o, observed_scores, sizeof(double) * n, cudaMemcpyHostToDevice, st));
    }
    if (innovations) {
        const int b = budget::resolve_bandwidth((long long)n, P.dependence_lag_hint);
        const size_t cnt = (size_t)std::max(1, P.num_null_draws) * m * (n + 2 * (size_t)b);
        RB_TRY(ar.alloc(&d_i, cnt));
        RB_CUDA(cudaMemcpyAsync(d_i, innovations, sizeof(double) * cnt, cudaMemcpyHostToDevice, st));
    }
    P.d_innovations = d_i;
    if (P.sample_offset < 0 || P.random_streams < 0 || P.random_streams > 1) return ST_INVALID;
    budget::Shard whole;
    const int status = budget::budget_core(d_c, (long long)m, (long long)n, d_o, P, whole, result, st);
    cudaStreamSynchronize(st);
    return status;
}

// Effective sample size of a host series (inference.py:446-501): returns n_eff, tau_int, lags used.
RB_API int rocco_effective_sample_size_f64(const double *values, size_t n, int max_lag, double *n_eff, double *tau_int, int *lags_used)
{
    if (!values || !n_eff || !tau_int || !lags_used) return ST_INVALID;
    *n_eff = (double)std::max<size_t>(1, n); *tau_int = 1.0; *lags_used = 0;
    if (n < 4) return 0;
    RB_TRY(ensure_device());
    HostScope lease;
    cudaStream_t st = lease.stream();
    Arena ar(st);
    double *d_v = nullptr;
    RB_TRY(ar.alloc(&d_v, n));
    RB_CUDA(cudaMemcpyAsync(d_v, values, sizeof(double) * n, cudaMemcpyHostToDevice, st));
    const double mean = numpy_sum_f64(values, n) / (double)n;                 // np.mean restated (the data is host-side already)
    if (!std::isfinite(mean)) return ST_NONFINITE;
    const int status = budget::effective_sample_size(ar, d_v, (long long)n, 0, 0.0, 1.0, mean, max_lag, n_eff, tau_int, lags_used, st);
    cudaStreamSynchronize(st);
    return status;
}

// Median and count of the strictly positive entries of a host score track (rocco.py:762-769); 1.0 / 0 when there are none.
RB_API int rocco_positive_score_median_f64(const double *scores, size_t n, double *median, long long *count)
{
    if (!scores || !median || !count) return ST_INVALID;
    *median = 1.0; *count = 0;
    if (n == 0) return 0;
    RB_TRY(ensure_device());
    HostScope lease;
    cudaStream_t st = lease.stream();
    Arena ar(st);
    double *d_s = nullptr, *d_sorted = nullptr, *d_out = nullptr;
    char *d_tmp = nullptr;
    RB_TRY(ar.alloc(&d_s, n));
    RB_TRY(ar.alloc(&d_sorted, n));
    RB_TRY(ar.alloc(&d_out, 2));
    RB_TRY(ar.alloc(&d_tmp, budget::sort_track_bytes((long long)n)));
    RB_CUDA(cudaMemcpyAsync(d_s, scores, sizeof(double) * n, cudaMemcpyHostToDevice, st));
    RB_TRY(budget::sort_track(d_tmp, d_s, d_sorted, (long long)n, st));
    budget::k_positive_median<<<1, 32, 0, st>>>(d_sorted, (long long)n, d_out);
    RB_LAUNCH_CHECK();
    double h[2];
    RB_CUDA(cudaMemcpyAsync(h, d_out, sizeof(h), cudaMemcpyDeviceToHost, st));
    RB_CUDA(cudaStreamSynchronize(st));
    *median = h[0];
    *count = (long long)h[1];
    return 0;
}

}  // extern "C"
