// Exact order statistics for the monotone variance trend WITHOUT sorting the row.
//
// The reference sorts the n (|signal|, variance) pairs of every sample row lexicographically
// (wls_backend.c:454), cuts them into B = max(4, floor(1 + log2(n+1))) equal-count bins and takes, per bin,
// the median |signal| by rank and the median variance (wls_backend.c:476-505).  Only ~3B order statistics
// per row are ever used, so the sort is replaced by a histogram multi-select:
//
//   T1  k_xhist      stream |C|: 16384 order-preserving buckets (1024 per octave of the bit pattern) per row
//   T2  k_xplan      per row: prefix sums -> bucket + in-bucket rank of every wanted x-rank; buckets holding a
//                    bin boundary or a median rank become "slots"
//   T3  k_xcollect   stream (|C|, V): pairs in slot buckets are collected; every other pair has a definite bin
//                    (its bucket lies inside one bin) and is counted in that bin's variance histogram
//   T4  k_xresolve   per (row, slot): sort the ~1e3 collected pairs lexicographically -> exact x medians; pairs of
//                    boundary buckets get their exact bin from their rank and join the variance histograms
//   T5  k_yplan      per row, per bin: locate the variance bucket(s) of the bin's median rank(s)
//   T6  k_ycollect   stream (|C|, V) once more: collect the variances of those buckets (plus boundary-slot pairs)
//   T7  k_yresolve   per row: sort the few collected variances per bin -> exact medians -> PAVA -> knots
//
// Any bucket larger than its capacity (massive ties, e.g. an all-zero matrix) flags the ROW, and flagged rows
// take the sort-based path in wls.cu, which is exact for any input.  Results are identical either way.
#include "common.cuh"
#include "select.cuh"
#include "score.cuh"
#include "trend.cuh"

#include <math.h>

#include <algorithm>

namespace rb {
namespace score {

constexpr int NBX = 16384;              // |signal| buckets, order preserving: a coarse region of 1024 buckets below a fine region
constexpr int NBX_LO = 1024;            // of 15360 buckets; values outside both land in the first / last bucket
constexpr int NBY = 1024;               // variance buckets centred on the row's sampled median variance
// Bucket geometry, chosen from the row length so that the fullest bucket stays under the slot capacity:
//   n <= 6 M bins : fine region 1024 per octave on [2^-8, 2^7),  coarse on [2^-24, 2^-8);  variances 64 per octave (16 octaves)
//   n  > 6 M bins : fine region 2048 per octave on [2^-6, 2^1.5), coarse 128 per octave on [2^-14, 2^-6); variances 128 per
//                   octave (8 octaves)
struct BucketGeom { int xshift; unsigned xb0; int xshift_lo; unsigned xb0_lo; int yshift; };
static BucketGeom bucket_geometry(long long n)
{
    if (n <= 6000000LL) return BucketGeom{42, (unsigned)(0x3F70000000000000ULL >> 42), 46, (unsigned)(0x3E70000000000000ULL >> 46), 46};
    return BucketGeom{41, (unsigned)(0x3F90000000000000ULL >> 41), 45, (unsigned)(0x3F10000000000000ULL >> 45), 45};
}
constexpr int YSAMPLE = 2048;
constexpr int MAXB = 32;                // bins per row (n < 2^31)
constexpr int MAXSLOT = 3 * MAXB;
constexpr int CAPX = 8192;              // pairs per x slot
constexpr int CAPY_MAX = 16384;         // variances per (bin, k) slot (TrendBuffers::capy)
constexpr int CHUNK = 131072;           // elements streamed per CTA
constexpr int ST_THREADS = 512;
int trend_fused_max_window() { return 1025; }

// The fine region carries the bulk of a row; the coarse one exists for rows with much mass near zero (a bootstrap
// draw  residual x multiplier  has a log-divergent density at 0), whose lowest equal-count bins end far below it.
__device__ __forceinline__ int xbucket(double x, const BucketGeom &G)
{
    const unsigned long long bits = (unsigned long long)__double_as_longlong(x);
    const int b = (int)(unsigned)(bits >> G.xshift) - (int)G.xb0;
    if (b >= 0) return min(NBX_LO + b, NBX - 1);
    const int t = (int)(unsigned)(bits >> G.xshift_lo) - (int)G.xb0_lo;
    return min(max(t, 0), NBX_LO - 1);
}
__device__ __forceinline__ int ybucket(double y, int yb0, const BucketGeom &G)
{
    const int u = (int)((unsigned long long)__double_as_longlong(y) >> G.yshift);
    const int b = u - yb0;
    return b < 0 ? 0 : (b >= NBY ? NBY - 1 : b);
}
// T3's 32-bit key of a pair, written by the fused rolling-variance pass: |signal| bucket << 18 | variance bits >> yshift.
// V is floored at 1e-8 (a NaN window gives the floor), so its sign bit is clear and a shift by 45 or 46 leaves at most
// 18 bits; T3 then finds both buckets of a pair without reading C or V (ybucket(v) == clamp((key & 0x3FFFF) - yb0)).
constexpr int KEY_YBITS = 18;
__device__ __forceinline__ unsigned pair_key(int xb, double v, const BucketGeom &G)
{
    return ((unsigned)xb << KEY_YBITS) | ((unsigned)__double2hiint(v) >> (G.yshift - 32));
}
__device__ __forceinline__ int bin_of_rank(long long p, long long N, int B)
{
    int b = (int)((p * B) / N);
    if (b >= B) b = B - 1;
    while (b + 1 < B && ((long long)(b + 1) * N) / B <= p) ++b;
    while (b > 0 && ((long long)b * N) / B > p) --b;
    return b;
}

enum FallbackReason { FB_XSLOT = 1, FB_XCOUNT = 2, FB_YTOTAL = 4, FB_YSLOT = 8, FB_YCOUNT = 16 };

struct RowPlan {
    int nslot;
    int fallback;                      // bit mask of FallbackReason
    int yb0;                           // variance bucket offset of this row
    int slot_bucket[MAXSLOT];
    int slot_prefix[MAXSLOT];          // rank of the first pair of the bucket
    int slot_count[MAXSLOT];
    int slot_boundary[MAXSLOT];        // number of bin boundaries inside the bucket
    int slot_brank[MAXSLOT];           // rank inside the slot of its (last) boundary: pairs below it belong to the lower bin
    int slot_done[MAXSLOT];            // resolved by the selection kernel (the sort kernels skip it)
    int ybin_done[MAXB];               // bin's variance medians resolved by the selection kernel
    // x medians: per bin up to two ranks -> (slot, rank inside slot)
    int xm_slot[MAXB][2];
    int xm_rank[MAXB][2];
    double xm_val[MAXB][2];
    // y medians: per bin up to two ranks -> (variance bucket, rank inside bucket)
    int ym_bucket[MAXB][2];
    int ym_rank[MAXB][2];
    int ym_count[MAXB][2];
    double ym_val[MAXB][2];
};

struct TrendBuffers {
    int *xhist;            // [m][NBX]
    unsigned char *lut;    // [m][NBX]  slot id or 0xFF
    unsigned char *binlo;  // [m][NBX]  bin of the bucket (valid when the bucket holds no boundary)
    RowPlan *plan;         // [m]
    double2 *cand;         // [m][MAXSLOT][CAPX]
    int *cand_cnt;         // [m][MAXSLOT]
    int *yhist;            // [m][MAXB][NBY]
    double *ycand;         // [m][MAXB][2][capy]
    int *ycand_cnt;        // [m][MAXB][2]
    unsigned long long *yover_min, *yover_max;   // [m][MAXB][2]  bit-pattern range of the variances that did not fit their slot
    unsigned short *codes;  // [m][code_stride]  T3 -> T6: bin << 10 | variance bucket of every pair (0xFFFF: not T6's business)
    unsigned *keys;         // [m][code_stride]  fused rolling variance -> T3: pair_key of every pair (fused pass only; nullptr: T3 reads C and V)
    long long code_stride;  // n rounded up to a multiple of 8 (128-bit loads)
    long long rows;
    BucketGeom geom;
    int capy;              // capacity of a ycand slot
};

// ------------------------------------------------------------------ T1
__global__ void __launch_bounds__(ST_THREADS) k_xhist(const double *__restrict__ C, long long n, long long row_stride, int *xhist, BucketGeom G)
{
    extern __shared__ int s_h[];
    const long long row = blockIdx.y;
    const long long c0 = (long long)blockIdx.x * CHUNK, c1 = min(n, c0 + CHUNK);
    for (int k = threadIdx.x; k < NBX; k += ST_THREADS) s_h[k] = 0;
    __syncthreads();
    const double *c = C + row * row_stride;
    for (long long j = c0 + threadIdx.x; j < c1; j += ST_THREADS) atomicAdd(&s_h[xbucket(fabs(c[j]), G)], 1);
    __syncthreads();
    int *g = xhist + row * NBX;
    for (int k = threadIdx.x; k < NBX; k += ST_THREADS) {
        const int v = s_h[k];
        if (v) atomicAdd(&g[k], v);
    }
}

// T3 runs on a PERSISTENT grid: the rows of the matrix, each padded to a multiple of 1024 pairs and laid end to end, are
// cut into gridDim.x equal contiguous ranges (multiples of 1024), so that a CTA sets up the per-row table and clears and
// flushes its 128 KB of histograms once per row it touches (one or two) instead of once per 131072 pairs, and no wave of
// CTAs is left partly filled.  (T1 and T6, whose per-CTA setup is small, were measured slower in this form -- 296
// separate streams instead of neighbouring chunks -- and keep one CTA per 131072-element chunk.)
__device__ __forceinline__ long long padded_row(long long n) { return (n + 1023) & ~1023LL; }
__device__ __forceinline__ void cta_range(long long rows, long long n, long long *g0, long long *g1)
{
    const long long total = rows * padded_row(n);
    long long per = (total + gridDim.x - 1) / gridDim.x;
    per = (per + 1023) & ~1023LL;
    *g0 = min(total, per * blockIdx.x);
    *g1 = min(total, *g0 + per);
}

// ------------------------------------------------------------------ T1 fused with the rolling AR(1) variance
// One CTA streams RV_CHUNK bins of one row in tiles of RV_T bins: the tile (+ w-1 halo) is staged in shared memory in a
// padded layout (position i + i/8, so that 8-bin-per-block accesses are bank-conflict free), every block of 8
// consecutive variances gets direct 31-term window sums for the first and sliding updates for the next 7 (far less
// drift than the reference's whole-row slide), each thread computes two such blocks with their dependent sum chains
// interleaved (worth 1.6 ms per step against one block per thread), results go back through shared memory for coalesced
// stores, and the same pass feeds the |C| histogram.  Replaces wls_backend.c:610-742 + the T1 pass.
// Staging is asynchronous and double-buffered: tile t+1 arrives by 8-byte cp.async copies (the padded layout keeps
// no 16-byte alignment) while tile t computes.  Interior tiles histogram each block's own 8 bins from the registers
// that hold them for the window sums; edge tiles (first / last of a row, a partial tail) read them back from shared
// memory.  The histogram keeps 16-bit counts, two buckets per word, so that two CTAs with two tile buffers each fit
// an SM and the barrier and store phases of one overlap the window arithmetic of the other.
// The pass also leaves T3 the pair_key of every bin, built from the bucket just counted and the
// variance just computed: interior tiles store each block's 8 keys as two 128-bit stores straight from registers (block
// starts are multiples of 8 bins, so 32-byte aligned), edge tiles one key per bin.
constexpr int RV_T = 4096;                   // bins per CTA iteration
constexpr int RV_K = 8;                      // outputs per block (direct window sums for the first, slides for the rest)
constexpr int RV_B = 2;                      // blocks per thread: blocks tid and tid + RV_THREADS, computed interleaved
constexpr int RV_THREADS = RV_T / (RV_K * RV_B);   // 256 at <= 128 registers: two CTAs per SM (32 KB histogram + two tile
                                                   // buffers of 37 KB at w = 31 each)
constexpr int RV_CHUNK = 15 * RV_T;          // bins per CTA: every bucket count fits the 16-bit halves of the shared histogram
static_assert(RV_CHUNK < 65536, "16-bit histogram counters");
constexpr int RV_MAXW = 1025;

__host__ __device__ __forceinline__ int padpos(int i) { return i + (i >> 3); }
// doubles per tile buffer (span <= RV_T + w - 1), even so that the second buffer starts 16-byte aligned
__host__ __device__ __forceinline__ int rv_buf(int w) { return (padpos(RV_T + w) + 1) & ~1; }

__device__ __forceinline__ void cp_async8(double *dst, const double *src)
{
    asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"((unsigned)__cvta_generic_to_shared(dst)), "l"(src) : "memory");
}

// W > 0: compile-time window (31 = the reference default): interior tiles run fully unrolled from registers.
template <int W>
__global__ void __launch_bounds__(RV_THREADS, 2) k_rollvar_xhist(const double *__restrict__ C, long long n, long long row_stride, int w_rt,
                                                               double *__restrict__ V, int *xhist, BucketGeom G,
                                                               unsigned *__restrict__ keys, long long key_stride)
{
    extern __shared__ int s_dyn[];
    const int w = W > 0 ? W : w_rt;
    unsigned *s_h = reinterpret_cast<unsigned *>(s_dyn);           // NBX / 2: bucket b counts in the 16-bit half b & 1 of word b / 2
    double *s_buf = reinterpret_cast<double *>(s_dyn + NBX / 2);  // 2 x rv_buf(w): tile t in buffer t & 1
    const long long row = blockIdx.y;
    const double *c = C + row * row_stride;
    double *v = V + row * row_stride;
    unsigned *const kr = keys + row * key_stride;
    const long long c0 = (long long)blockIdx.x * RV_CHUNK, c1 = min(n, c0 + RV_CHUNK);
    const long long half = w / 2, last = n - w;
    const double wd = (double)w, pairs = (double)(w - 1), rwd = 1.0 / wd, shrink = 1.0 + 1.0 / (wd + 1.0) + 1.0e-4;      // c1 of ar1_window_variance
    const int tid = threadIdx.x;
    auto count = [&](double x) { const int b = xbucket(fabs(x), G); atomicAdd(&s_h[b >> 1], 1u << ((b & 1) << 4)); return b; };
    const int bstride = rv_buf(w);
    // staged range of the tile starting at j0: [tlo, tlo + span)
    auto tile_range = [&](long long j0, long long *tlo, int *span) {
        const long long j1 = min(c1, j0 + RV_T);
        long long lo = j0 - half; if (lo < 0) lo = 0; else if (lo > last) lo = last;
        long long hi = (j1 - 1) - half; if (hi < 0) hi = 0; else if (hi > last) hi = last;
        *tlo = lo;
        *span = (int)(hi - lo) + w;
    };
    auto stage = [&](long long j0, double *buf) {
        long long tlo; int span;
        tile_range(j0, &tlo, &span);
        const double *src = c + tlo;
#pragma unroll 4
        for (int e = tid; e < span; e += RV_THREADS) cp_async8(buf + padpos(e), src + e);
        asm volatile("cp.async.commit_group;" ::: "memory");
    };
    double *s_in = s_buf, *s_next = s_buf + bstride;
    stage(c0, s_in);
    for (int k = tid; k < NBX / 2; k += RV_THREADS) s_h[k] = 0;
    for (long long j0 = c0; j0 < c1; j0 += RV_T) {
        const long long j1 = min(c1, j0 + RV_T);
        long long tlo; int span;
        tile_range(j0, &tlo, &span);
        asm volatile("cp.async.wait_group 0;" ::: "memory");
        __syncthreads();                                           // this tile has landed; the other buffer has been copied out
        if (j0 + RV_T < c1) stage(j0 + RV_T, s_next);
        const bool interior = (j0 - half >= 0) && ((j1 - 1) - half <= last) && (j1 - j0 == RV_T);
        double res[RV_B][RV_K];
        if (W > 0 && interior) {
            // window of output k of block b starts at staged position b*8 + k; padded address = b*9 + q + (q >> 3).  The
            // blocks' sums are independent chains, interleaved here so that each thread keeps RV_B of them in flight.
            double y[RV_B][W + RV_K - 1];
#pragma unroll
            for (int h = 0; h < RV_B; ++h) {
                const double *base = s_in + (tid + h * RV_THREADS) * 9;
#pragma unroll
                for (int q = 0; q < W + RV_K - 1; ++q) y[h][q] = base[q + (q >> 3)];
            }
            double s1[RV_B], s2[RV_B], sl[RV_B];
#pragma unroll
            for (int h = 0; h < RV_B; ++h) s1[h] = s2[h] = sl[h] = 0.0;
#pragma unroll
            for (int q = 0; q < W; ++q) {
#pragma unroll
                for (int h = 0; h < RV_B; ++h) {
                    s1[h] = __dadd_rn(s1[h], y[h][q]);
                    s2[h] = __fma_rn(y[h][q], y[h][q], s2[h]);
                    if (q + 1 < W) sl[h] = __fma_rn(y[h][q], y[h][q + 1], sl[h]);
                }
            }
#pragma unroll
            for (int k = 0; k < RV_K; ++k) {
#pragma unroll
                for (int h = 0; h < RV_B; ++h) {
                    if (k > 0) {
                        const double out_v = y[h][k - 1], nx = y[h][k - 1 + W];
                        s1[h] = __dadd_rn(__dsub_rn(s1[h], out_v), nx);
                        s2[h] = __fma_rn(nx, nx, __fma_rn(-out_v, out_v, s2[h]));
                        sl[h] = __fma_rn(y[h][k - 2 + W], nx, __fma_rn(-out_v, y[h][k], sl[h]));
                    }
                    const double cur = ar1_window_variance(s1[h], s2[h], sl[h], y[h][k], y[h][k + W - 1], wd, rwd, pairs, shrink);
                    res[h][k] = dmax(cur, 1.0e-8);                                 // wls_backend.c:869
                }
            }
            // own bins (staged b*8 + half + k): histogram, and the keys four at a time so that no more than four are live
#pragma unroll
            for (int h = 0; h < RV_B; ++h)
#pragma unroll
                for (int k4 = 0; k4 < RV_K; k4 += 4) {
                    unsigned kk[4];
#pragma unroll
                    for (int q = 0; q < 4; ++q) kk[q] = pair_key(count(y[h][W / 2 + k4 + q]), res[h][k4 + q], G);
                    *reinterpret_cast<uint4 *>(kr + j0 + (tid + h * RV_THREADS) * RV_K + k4) = make_uint4(kk[0], kk[1], kk[2], kk[3]);
                }
        } else {
#pragma unroll
          for (int h = 0; h < RV_B; ++h) {
            const long long jt = j0 + (long long)(tid + h * RV_THREADS) * RV_K;
            double s1 = 0.0, s2 = 0.0, sl = 0.0, cur = 0.0;
            long long tprev = -1;
#pragma unroll
            for (int k = 0; k < RV_K; ++k) {
                const long long j = jt + k;
                res[h][k] = 0.0;
                if (j >= j1) continue;
                long long t = j - half;
                if (t < 0) t = 0; else if (t > last) t = last;
                const int r = (int)(t - tlo);
                if (t != tprev) {
                    if (tprev < 0) {
                        s1 = s2 = sl = 0.0;
                        double a = s_in[padpos(r)];
                        for (int q = 0; q < w; ++q) {
                            const double nx = (q + 1 < w) ? s_in[padpos(r + q + 1)] : 0.0;
                            s1 = __dadd_rn(s1, a);
                            s2 = __fma_rn(a, a, s2);
                            if (q + 1 < w) sl = __fma_rn(a, nx, sl);
                            a = nx;
                        }
                    } else {
                        const double out_v = s_in[padpos(r - 1)], nx = s_in[padpos(r - 1 + w)];
                        const double lag_l = s_in[padpos(r - 1 + w - 1)], lag_r = s_in[padpos(r)];
                        s1 = __dadd_rn(__dsub_rn(s1, out_v), nx);
                        s2 = __fma_rn(nx, nx, __fma_rn(-out_v, out_v, s2));
                        sl = __fma_rn(lag_l, nx, __fma_rn(-out_v, lag_r, sl));
                    }
                    cur = ar1_window_variance(s1, s2, sl, s_in[padpos(r)], s_in[padpos(r + w - 1)], wd, rwd, pairs, shrink);
                    tprev = t;
                }
                res[h][k] = dmax(cur, 1.0e-8);
            }
#pragma unroll
            for (int k = 0; k < RV_K; ++k)
                if (jt + k < j1) {
                    const int b = count(s_in[padpos((int)(jt + k - tlo))]);
                    kr[jt + k] = pair_key(b, res[h][k], G);
                }
          }
        }
        __syncthreads();                                           // every window has been read: the slots can take the results
        double *const s_out = s_in;
#pragma unroll
        for (int h = 0; h < RV_B; ++h) {
            double *ob = s_out + (tid + h * RV_THREADS) * 9;       // padpos(b * 8 + k) = b * 9 + k
#pragma unroll
            for (int k = 0; k < RV_K; ++k) ob[k] = res[h][k];
        }
        __syncthreads();
        // plain stores: nothing waits for them; the next iteration's barrier orders these shared reads before the
        // buffer is staged again
        double *dst = v + j0;
        for (int e = tid; e < (int)(j1 - j0); e += RV_THREADS) dst[e] = s_out[padpos(e)];
        double *const t = s_in; s_in = s_next; s_next = t;
    }
    int *g = xhist + row * NBX;
    for (int k = tid; k < NBX / 2; k += RV_THREADS) {
        const unsigned val = s_h[k];
        if (val & 0xFFFFu) atomicAdd(&g[2 * k], (int)(val & 0xFFFFu));
        if (val >> 16) atomicAdd(&g[2 * k + 1], (int)(val >> 16));
    }
}

// ------------------------------------------------------------------ T2
__global__ void __launch_bounds__(256) k_xplan(TrendBuffers T, const double *__restrict__ V, long long row_stride, long long n, int B)
{
    extern __shared__ int s_plan[];
    int *s_pre = s_plan;                 // NBX + 1
    int *s_part = s_plan + NBX + 1;      // 256
    const long long row = blockIdx.x;
    const int *h = T.xhist + row * NBX;
    // exclusive prefix over NBX buckets: 64 consecutive buckets per thread
    const int per = NBX / 256;
    int loc = 0;
    for (int k = 0; k < per; ++k) loc += h[threadIdx.x * per + k];
    s_part[threadIdx.x] = loc;
    __syncthreads();
    if (threadIdx.x == 0) {
        int acc = 0;
        for (int t = 0; t < 256; ++t) { const int v = s_part[t]; s_part[t] = acc; acc += v; }
    }
    __syncthreads();
    {
        int acc = s_part[threadIdx.x];
        for (int k = 0; k < per; ++k) { s_pre[threadIdx.x * per + k] = acc; acc += h[threadIdx.x * per + k]; }
        if (threadIdx.x == 255) s_pre[NBX] = acc;
    }
    __syncthreads();
    unsigned char *lut = T.lut + row * NBX, *binlo = T.binlo + row * NBX;
    // bin of every bucket's first rank = number of bin boundaries floor(b n / B), b = 1..B-1, at or below it
    __shared__ long long s_lo[MAXB];
    if (threadIdx.x < B) s_lo[threadIdx.x] = ((long long)threadIdx.x * n) / B;
    __syncthreads();
    for (int k = threadIdx.x; k < NBX; k += 256) {
        lut[k] = 0xFF;
        const long long r = min((long long)s_pre[k], n - 1);
        int bin = 0;
        for (int b = 1; b < B; ++b) bin += (s_lo[b] <= r);
        binlo[k] = (unsigned char)bin;
    }
    __syncthreads();
    // centre the variance buckets on the median of a strided sample of this row's variances (a radix select: the bit
    // patterns of positive doubles order like the values)
    {
        unsigned long long *s_smp = reinterpret_cast<unsigned long long *>(s_plan + NBX + 1 + 256 + 1);   // 8-byte aligned: NBX+258 ints
        const int take = (int)min((long long)YSAMPLE, n);
        for (int k = threadIdx.x; k < take; k += 256) {
            const long long i = (n <= YSAMPLE) ? k : (long long)(((double)k + 0.5) * ((double)n / (double)YSAMPLE));
            s_smp[k] = (unsigned long long)__double_as_longlong(V[row * row_stride + min(i, n - 1)]);
        }
        __syncthreads();
        const unsigned long long med = block_select<256>(s_smp, take, take / 2, nullptr, 0ULL, plan_scratch(s_smp + YSAMPLE), nullptr, nullptr);
        if (threadIdx.x == 0) T.plan[row].yb0 = (int)(med >> T.geom.yshift) - NBY / 2;
        __syncthreads();
    }
    // the <= 3B wanted ranks (bin boundary, upper median, lower median) are located in parallel, one thread each; slots
    // are then handed out by one thread in the fixed order boundary, median 1, median 0 per bin (deterministic slot ids)
    __shared__ int s_req_bucket[3 * MAXB];
    __shared__ int s_req_rank[3 * MAXB];
    RowPlan &P = T.plan[row];
    for (int q = threadIdx.x; q < 3 * B; q += 256) {
        const int b = q / 3, kind = q % 3;                  // 0: boundary at the bin's first rank, 1: upper median, 2: lower median
        const long long lo = ((long long)b * n) / B, hi = ((long long)(b + 1) * n) / B;
        const long long w = hi - lo;
        long long r = -1;
        if (w > 0) {
            if (kind == 0) r = b > 0 ? lo : -1;
            else if (kind == 1) r = lo + w / 2;
            else r = (w & 1) == 0 ? lo + w / 2 - 1 : -1;
        }
        int bucket = -1;
        if (r >= 0) {                                       // largest bucket with pre[bucket] <= r
            int l = 0, h = NBX;
            while (h - l > 1) { const int mid = (l + h) >> 1; if ((long long)s_pre[mid] <= r) l = mid; else h = mid; }
            bucket = l;
        }
        s_req_bucket[q] = bucket;
        s_req_rank[q] = bucket >= 0 ? (int)(r - s_pre[bucket]) : 0;
    }
    __syncthreads();
    if (threadIdx.x != 0) return;
    P.nslot = 0; P.fallback = 0;
    auto slot_for = [&](int b) {
        int sl = lut[b];
        if (sl == 0xFF) {
            sl = P.nslot++;
            lut[b] = (unsigned char)sl;
            P.slot_bucket[sl] = b; P.slot_prefix[sl] = s_pre[b]; P.slot_count[sl] = s_pre[b + 1] - s_pre[b];
            P.slot_boundary[sl] = 0; P.slot_brank[sl] = 0; P.slot_done[sl] = 0;
            if (P.slot_count[sl] > CAPX) P.fallback |= FB_XSLOT;
        }
        return sl;
    };
    for (int b = 0; b < B; ++b) {
        for (int k = 0; k < 2; ++k) { P.xm_slot[b][k] = -1; P.xm_rank[b][k] = 0; P.ym_bucket[b][k] = -1; }
        P.ybin_done[b] = 0;
        if (s_req_bucket[3 * b] >= 0) {
            const int sl = slot_for(s_req_bucket[3 * b]);
            P.slot_boundary[sl] += 1; P.slot_brank[sl] = s_req_rank[3 * b];
        }
        if (s_req_bucket[3 * b + 1] >= 0) { P.xm_slot[b][1] = slot_for(s_req_bucket[3 * b + 1]); P.xm_rank[b][1] = s_req_rank[3 * b + 1]; }
        if (s_req_bucket[3 * b + 2] >= 0) { P.xm_slot[b][0] = slot_for(s_req_bucket[3 * b + 2]); P.xm_rank[b][0] = s_req_rank[3 * b + 2]; }
    }
}

// ------------------------------------------------------------------ T3
// One 16-bit entry per |signal| bucket for the two streaming passes: the bucket's bin (5 bits), whether it holds a bin
// boundary (bit 7), and its slot (0xFF: none) -- a single shared-memory load per pair.
__device__ __forceinline__ void bucket_table(unsigned short *s_tab, const unsigned char *lut, const unsigned char *binlo, const RowPlan &P,
                                             int threads)
{
    for (int k = threadIdx.x; k < NBX; k += threads) {
        const unsigned sl = lut[k];
        const unsigned bnd = (sl != 0xFFu && P.slot_boundary[sl] != 0) ? 0x80u : 0u;
        s_tab[k] = (unsigned short)((unsigned)binlo[k] | bnd | (sl << 8));
    }
}
constexpr int XC_THREADS = 1024;          // one CTA per SM (160 KB of histograms + LUTs): 32 warps hide the LUT/atomic chain

__global__ void __launch_bounds__(XC_THREADS) k_xcollect(const double *__restrict__ C, const double *__restrict__ V, long long n,
                                                         long long row_stride, TrendBuffers T, int B)
{
    extern __shared__ int s_raw[];
    int *s_yh = s_raw;                                              // [B][NBY]
    unsigned short *s_tab = reinterpret_cast<unsigned short *>(s_raw + B * NBY);    // per |signal| bucket: bin | boundary << 7 | slot << 8
    long long g0, g1;
    cta_range(T.rows, n, &g0, &g1);
    const long long np = padded_row(n);
    for (long long g = g0; g < g1;) {
        const long long row = g / np, c0 = g - row * np, seg = min(np - c0, g1 - g), c1 = min(n, c0 + seg);
        g += seg;
        const RowPlan &P = T.plan[row];
        if (P.fallback || c0 >= c1) continue;
        __syncthreads();                                            // the previous row's flush is done
        for (int k = threadIdx.x; k < B * NBY; k += XC_THREADS) s_yh[k] = 0;
        bucket_table(s_tab, T.lut + row * NBX, T.binlo + row * NBX, P, XC_THREADS);
        __syncthreads();
        const double *c = C + row * row_stride, *v = V + row * row_stride;
        double2 *cand = T.cand + (size_t)row * MAXSLOT * CAPX;
        int *ccnt = T.cand_cnt + row * MAXSLOT;
        unsigned short *codes = T.codes + row * T.code_stride;
        const int yb0 = P.yb0;
        // eight independent loads in flight per thread, then the table lookups, then the slot counters (independent global
        // atomics, all in flight together), and only then the stores and histogram updates that depend on them
        constexpr int U = 8;
        for (long long jb = c0; jb < c1; jb += U * XC_THREADS) {
            double xs[U], ys[U];
#pragma unroll
            for (int u = 0; u < U; ++u) {
                const long long j = jb + u * XC_THREADS + threadIdx.x;
                xs[u] = (j < c1) ? fabs(c[j]) : -1.0;
                ys[u] = (j < c1) ? v[j] : 0.0;
            }
            unsigned es[U];
            int pos[U];
#pragma unroll
            for (int u = 0; u < U; ++u) es[u] = (xs[u] < 0.0) ? 0xFFFFFFFFu : (unsigned)s_tab[xbucket(xs[u], T.geom)];
#pragma unroll
            for (int u = 0; u < U; ++u) pos[u] = (es[u] < 0xFF00u) ? atomicAdd(&ccnt[es[u] >> 8], 1) : CAPX;   // slot bucket (~2 % of the pairs)
#pragma unroll
            for (int u = 0; u < U; ++u) {
                const unsigned e = es[u];
                if (e == 0xFFFFFFFFu) continue;
                unsigned short code = 0xFFFFu;
                if (e < 0xFF00u && pos[u] < CAPX) cand[(size_t)(e >> 8) * CAPX + pos[u]] = make_double2(xs[u], ys[u]);
                if (!(e < 0xFF00u && (e & 0x80u))) {                // (boundary bucket: its bin is settled by T4)
                    const int bin = (int)(e & 31u), yb = ybucket(ys[u], yb0, T.geom);
                    atomicAdd(&s_yh[bin * NBY + yb], 1);
                    code = (unsigned short)((bin << 10) | yb);
                }
                codes[jb + u * XC_THREADS + threadIdx.x] = code;    // T6 reads two bytes per pair instead of sixteen
            }
        }
        __syncthreads();
        int *gh = T.yhist + (size_t)row * MAXB * NBY;
        for (int k = threadIdx.x; k < B * NBY; k += XC_THREADS) {
            const int val = s_yh[k];
            if (val) atomicAdd(&gh[k], val);
        }
    }
}

// T3 from the keys the fused rolling-variance pass left (pair_key): 4 bytes per pair instead of C and V's 16, no
// per-pair bucketing of doubles, and C and V gathered only for the pairs of slot buckets (~2 %).  The same histogram
// updates, codes and candidates as k_xcollect.  A thread takes groups of four consecutive pairs -- one 128-bit key load,
// one 64-bit store of their codes -- XK_R groups 4 * XC_THREADS pairs apart.  Ranges start at a multiple of 1024 pairs
// and end at one or at n, so a group never straddles two CTAs; keys at or past c1 are row padding and are masked.
constexpr int XK_R = 2;

__global__ void __launch_bounds__(XC_THREADS) k_xcollect_keys(const double *__restrict__ C, const double *__restrict__ V, long long n,
                                                              long long row_stride, TrendBuffers T, int B)
{
    extern __shared__ int s_raw[];
    int *s_yh = s_raw;                                              // [B][NBY]
    unsigned short *s_tab = reinterpret_cast<unsigned short *>(s_raw + B * NBY);    // per |signal| bucket: bin | boundary << 7 | slot << 8
    long long g0, g1;
    cta_range(T.rows, n, &g0, &g1);
    const long long np = padded_row(n);
    for (long long g = g0; g < g1;) {
        const long long row = g / np, c0 = g - row * np, seg = min(np - c0, g1 - g), c1 = min(n, c0 + seg);
        g += seg;
        const RowPlan &P = T.plan[row];
        if (P.fallback || c0 >= c1) continue;
        __syncthreads();                                            // the previous row's flush is done
        for (int k = threadIdx.x; k < B * NBY; k += XC_THREADS) s_yh[k] = 0;
        bucket_table(s_tab, T.lut + row * NBX, T.binlo + row * NBX, P, XC_THREADS);
        __syncthreads();
        const double *c = C + row * row_stride, *v = V + row * row_stride;
        const unsigned *keys = T.keys + row * T.code_stride;
        double2 *cand = T.cand + (size_t)row * MAXSLOT * CAPX;
        int *ccnt = T.cand_cnt + row * MAXSLOT;
        unsigned short *codes = T.codes + row * T.code_stride;
        const int yb0 = P.yb0;
        constexpr int U = 4 * XK_R;
        constexpr long long STEP = 4LL * XC_THREADS * XK_R;
        // Software-pipelined over iterations so that no iteration waits on a global round trip: the keys of iteration
        // i + 1 are loaded during iteration i, and a thread's first two slot pairs of iteration i (~2 % of the pairs: some
        // lane of a warp nearly always has one) get their slot counters bumped and their C and V gathered at the top of
        // iteration i + 1, to be filed at its end.  A third or later slot pair of one iteration (rows with heavy ties) is
        // filed on the spot after the loop body.
        auto load_keys = [&](long long jb0, uint4 *ks) {
#pragma unroll
            for (int r = 0; r < XK_R; ++r) {
                const long long jb = jb0 + 4LL * XC_THREADS * r;
                ks[r] = jb < c1 ? *reinterpret_cast<const uint4 *>(keys + jb) : make_uint4(0u, 0u, 0u, 0u);
            }
        };
        auto file_pair = [&](int off, unsigned sl) {               // one slot pair, filed with its own round trip
            const long long j = c0 + off;
            const int p = atomicAdd(&ccnt[sl], 1);
            if (p < CAPX) cand[(size_t)sl * CAPX + p] = make_double2(fabs(c[j]), v[j]);
        };
        uint4 kn[XK_R];
        load_keys(c0 + 4LL * threadIdx.x, kn);
        int oc0 = -1, oc1 = -1;                                     // carried slot pairs: offset from c0 (-1: none), slot
        unsigned sc0 = 0u, sc1 = 0u;
        for (long long jb0 = c0 + 4LL * threadIdx.x; jb0 < c1; jb0 += STEP) {
            uint4 ks[XK_R];
#pragma unroll
            for (int r = 0; r < XK_R; ++r) ks[r] = kn[r];
            load_keys(jb0 + STEP, kn);
            int pc0 = CAPX, pc1 = CAPX;
            double xc0 = 0.0, yc0 = 0.0, xc1 = 0.0, yc1 = 0.0;
            if (oc0 >= 0) { pc0 = atomicAdd(&ccnt[sc0], 1); xc0 = fabs(c[c0 + oc0]); yc0 = v[c0 + oc0]; }
            if (oc1 >= 0) { pc1 = atomicAdd(&ccnt[sc1], 1); xc1 = fabs(c[c0 + oc1]); yc1 = v[c0 + oc1]; }
            const int o = (int)(jb0 - c0);
            auto off_at = [&](int u) { return o + 4 * XC_THREADS * (u >> 2) + (u & 3); };
            int na = 0, on0 = -1, on1 = -1;
            unsigned sn0 = 0u, sn1 = 0u, more = 0u;
            unsigned cw[XK_R][2];
#pragma unroll
            for (int u = 0; u < U; ++u) {
                const int r = u >> 2, q = u & 3;
                const unsigned key = q == 0 ? ks[r].x : q == 1 ? ks[r].y : q == 2 ? ks[r].z : ks[r].w;
                unsigned code = 0xFFFFu;
                if (jb0 + 4LL * XC_THREADS * r + q < c1) {
                    const unsigned e = s_tab[key >> KEY_YBITS];
                    const bool slot = e < 0xFF00u;
                    if (slot) {
                        const unsigned sl = e >> 8;
                        if (na == 0) { on0 = off_at(u); sn0 = sl; }
                        else if (na == 1) { on1 = off_at(u); sn1 = sl; }
                        else more |= 1u << u;
                        ++na;
                    }
                    if (!(slot && (e & 0x80u))) {                   // (boundary bucket: its bin is settled by T4)
                        const unsigned bin = e & 31u;
                        const unsigned yb = (unsigned)min(max((int)(key & ((1u << KEY_YBITS) - 1u)) - yb0, 0), NBY - 1);
                        atomicAdd(&s_yh[bin * NBY + yb], 1);
                        code = (bin << 10) | yb;
                    }
                }
                unsigned &word = cw[r][(u >> 1) & 1];
                word = (u & 1) ? (word | (code << 16)) : code;
            }
#pragma unroll
            for (int r = 0; r < XK_R; ++r) {
                const long long jb = jb0 + 4LL * XC_THREADS * r;
                if (jb < c1) *reinterpret_cast<uint2 *>(codes + jb) = make_uint2(cw[r][0], cw[r][1]);
            }
            if (pc0 < CAPX) cand[(size_t)sc0 * CAPX + pc0] = make_double2(xc0, yc0);
            if (pc1 < CAPX) cand[(size_t)sc1 * CAPX + pc1] = make_double2(xc1, yc1);
            for (; more; more &= more - 1) {                        // (the slot is looked up again from the key)
                const int off = off_at(__ffs(more) - 1);
                file_pair(off, (unsigned)s_tab[keys[c0 + off] >> KEY_YBITS] >> 8);
            }
            oc0 = on0; sc0 = sn0; oc1 = on1; sc1 = sn1;
        }
        if (oc0 >= 0) file_pair(oc0, sc0);                          // the last iteration's carried pairs
        if (oc1 >= 0) file_pair(oc1, sc1);
        __syncthreads();
        int *gh = T.yhist + (size_t)row * MAXB * NBY;
        for (int k = threadIdx.x; k < B * NBY; k += XC_THREADS) {
            const int val = s_yh[k];
            if (val) atomicAdd(&gh[k], val);
        }
    }
}

// ------------------------------------------------------------------ T4 by selection (block_select: select.cuh)

// (row, slot) CTAs for the slots the selection handles: at most two median ranks and no boundary, or exactly one
// boundary and no median rank.  Everything else (short rows where a bucket spans several bins) is left to the sort
// kernels below.  A boundary slot is PARTITIONED in place around its boundary pair -- lexicographic (|signal|, variance)
// order, like the reference's comparator (wls_backend.c:207-230) -- which is all T6 needs: the first slot_brank pairs
// belong to the lower bin, the rest to the upper one.
template <int THREADS, int CAP_LO, int CAP_HI>
__global__ void __launch_bounds__(THREADS, 1024 / THREADS) k_xselect(TrendBuffers T, long long n, int B)
{
    extern __shared__ unsigned long long s_sel[];         // x keys [cap], then y keys [cap] for boundary slots
    __shared__ SelScratch S;
    __shared__ int s_want[4], s_nwant, s_cursor[2];
    const long long row = blockIdx.y;
    const int s = blockIdx.x;
    RowPlan &P = T.plan[row];
    if (P.fallback || s >= P.nslot) return;
    const int total = P.slot_count[s];
    if (total <= CAP_LO || total > CAP_HI) return;                               // not this tier
    const int cnt = min(T.cand_cnt[row * MAXSLOT + s], CAPX);
    if (cnt != total) return;                                                    // the sort kernel reports the mismatch
    const int nb = P.slot_boundary[s];
    if (threadIdx.x == 0) s_nwant = 0;
    __syncthreads();
    for (int q = threadIdx.x; q < 2 * B; q += THREADS)
        if (P.xm_slot[q >> 1][q & 1] == s) { const int w = atomicAdd(&s_nwant, 1); if (w < 4) s_want[w] = q; }
    __syncthreads();
    const int nwant = s_nwant;
    const bool median_only = (nb == 0 && nwant >= 1 && nwant <= 2);
    const bool boundary_only = (nb == 1 && nwant == 0);
    if (!median_only && !boundary_only) return;
    double2 *cand = T.cand + ((size_t)row * MAXSLOT + s) * CAPX;
    unsigned long long *kx = s_sel, *ky = s_sel + CAP_HI;
    for (int k = threadIdx.x; k < cnt; k += THREADS) {
        const double2 pr = cand[k];
        kx[k] = (unsigned long long)__double_as_longlong(pr.x);                  // |signal| >= 0, variance > 0: the bit patterns order like the values
        if (boundary_only) ky[k] = (unsigned long long)__double_as_longlong(pr.y);
    }
    __syncthreads();
    if (median_only) {
        for (int w = 0; w < nwant; ++w) {
            const int q = s_want[w];
            const unsigned long long key = block_select<THREADS>(kx, cnt, P.xm_rank[q >> 1][q & 1], nullptr, 0ULL, S, nullptr, nullptr);
            if (threadIdx.x == 0) P.xm_val[q >> 1][q & 1] = __longlong_as_double((long long)key);
        }
        if (threadIdx.x == 0) P.slot_done[s] = 1;
        return;
    }
    // boundary slot: the pair of rank rb is the first pair of the upper bin
    const int rb = P.slot_brank[s];
    int xbelow = 0, xequal = 0, ybelow = 0;
    const unsigned long long px = block_select<THREADS>(kx, cnt, rb, nullptr, 0ULL, S, &xbelow, &xequal);
    unsigned long long py = 0ULL;
    if (xequal > 1) py = block_select<THREADS>(ky, cnt, rb - xbelow, kx, px, S, &ybelow, nullptr);
    // lower bin: pairs lexicographically below the pivot, plus as many pivot-equal pairs as are needed to reach rb
    const int n_less = xbelow + ybelow;
    if (threadIdx.x == 0) { s_cursor[0] = 0; s_cursor[1] = 0; s_want[0] = rb - n_less; }
    __syncthreads();
    const long long pre = P.slot_prefix[s];
    const int bin_hi = bin_of_rank(pre + rb, n, B), bin_lo = bin_hi - 1;
    int *g = T.yhist + (size_t)row * MAXB * NBY;
    for (int k = threadIdx.x; k < cnt; k += THREADS) {
        const unsigned long long x = kx[k], y = ky[k];
        bool lower;
        if (x != px) lower = x < px;
        else if (xequal == 1) lower = false;                                     // the pivot itself
        else if (y != py) lower = y < py;
        else lower = atomicSub(&s_want[0], 1) > 0;                                // identical pairs are interchangeable
        const int pos = lower ? atomicAdd(&s_cursor[0], 1) : rb + atomicAdd(&s_cursor[1], 1);
        const double yv = __longlong_as_double((long long)y);
        cand[pos] = make_double2(__longlong_as_double((long long)x), yv);
        atomicAdd(&g[(lower ? bin_lo : bin_hi) * NBY + ybucket(yv, P.yb0, T.geom)], 1);
    }
    if (threadIdx.x == 0) P.slot_done[s] = 1;
}

// (bin, row) CTAs: the one or two median ranks of the bin's variances, selected from the collected bucket(s).  A bucket
// that outgrew its slot is still exact when every value in it is the same (variances sitting on the 1e-8 floor): the
// overflow's min / max were tracked by T6.
template <int THREADS, int CAP_LO, int CAP_HI>
__global__ void __launch_bounds__(THREADS, CAP_HI <= 4096 ? 1024 / THREADS : 1) k_yselect(TrendBuffers T, long long n, int B)
{
    extern __shared__ unsigned long long s_sel[];
    __shared__ SelScratch S;
    const long long row = blockIdx.y;
    const int b = blockIdx.x;
    RowPlan &P = T.plan[row];
    if (P.fallback) return;
    const long long lo = ((long long)b * n) / B, hi = ((long long)(b + 1) * n) / B;
    if (hi <= lo) return;
    {   // two launches share the bins by the size of their candidate lists: the small tier keeps several CTAs per SM
        int mx = 0;
        for (int k = 0; k < 2; ++k)
            if (P.ym_bucket[b][k] >= 0) mx = max(mx, min(T.ycand_cnt[((size_t)row * MAXB + b) * 2 + k], T.capy));
        if (mx <= CAP_LO || mx > CAP_HI) return;
    }
    double ym[2] = {0.0, 0.0};
    bool ok = true;
    for (int k = 1; k >= 0 && ok; --k) {
        if (P.ym_bucket[b][k] < 0) continue;
        if (k == 0 && P.ym_bucket[b][0] == P.ym_bucket[b][1]) continue;                 // resolved together with k = 1
        const size_t slot = ((size_t)row * MAXB + b) * 2 + k;
        const int total = T.ycand_cnt[slot];
        if (total != P.ym_count[b][k]) { ok = false; break; }                           // the sort kernel reports it
        const int cnt = min(total, T.capy);
        const double *src = T.ycand + slot * T.capy;
        for (int q = threadIdx.x; q < cnt; q += THREADS) s_sel[q] = (unsigned long long)__double_as_longlong(src[q]);
        __syncthreads();
        const bool same_bucket = (k == 1 && P.ym_bucket[b][0] == P.ym_bucket[b][1]);
        if (total > T.capy) {
            // over capacity: exact only if stored values and overflow are all one value
            int below = 0, equal = 0;
            const unsigned long long v = block_select<THREADS>(s_sel, cnt, 0, nullptr, 0ULL, S, &below, &equal);
            if (equal == cnt && T.yover_min[slot] == v && T.yover_max[slot] == v) {
                ym[k] = __longlong_as_double((long long)v);
                if (same_bucket) ym[0] = ym[k];
            } else ok = false;
        } else {
            ym[k] = __longlong_as_double((long long)block_select<THREADS>(s_sel, cnt, P.ym_rank[b][k], nullptr, 0ULL, S, nullptr, nullptr));
            if (same_bucket) ym[0] = __longlong_as_double((long long)block_select<THREADS>(s_sel, cnt, P.ym_rank[b][0], nullptr, 0ULL, S, nullptr, nullptr));
        }
        __syncthreads();
    }
    if (threadIdx.x == 0) {
        if (ok) { P.ym_val[b][0] = ym[0]; P.ym_val[b][1] = ym[1]; P.ybin_done[b] = 1; }
    }
}

// ------------------------------------------------------------------ T4
__device__ __forceinline__ bool pair_gt(const double2 &a, const double2 &b) { return a.x > b.x || (a.x == b.x && a.y > b.y); }

// Two tiers over the same slots: <256 threads, slots of <= 2048 pairs> (32 KB of shared memory, several CTAs per SM --
// almost every slot) and <512 threads, up to CAPX pairs> for the rare large ones; a CTA exits if the slot is not its tier.
template <int THREADS, int CAP_LO, int CAP_HI>
__device__ void xresolve_slot(TrendBuffers &T, long long n, int B, long long row, int s, double2 *s_p)
{
    constexpr int ST_THREADS = THREADS;
    RowPlan &P = T.plan[row];
    if (s >= P.nslot) return;
    const int cnt = min(T.cand_cnt[row * MAXSLOT + s], CAPX);
    if (P.slot_count[s] <= CAP_LO || P.slot_count[s] > CAP_HI) return;          // not this tier
    if (P.slot_done[s]) return;                                                 // resolved by k_xselect
    if (cnt != P.slot_count[s]) { if (threadIdx.x == 0) atomicOr(&P.fallback, FB_XCOUNT); return; }
    int len = 1;
    while (len < cnt) len <<= 1;
    double2 *cand = T.cand + ((size_t)row * MAXSLOT + s) * CAPX;
    if (!P.slot_boundary[s]) {
        // median-only slot: only the |signal| value at one or two ranks is wanted, so the keys are sorted alone (half the
        // shared-memory traffic of the pair sort, one compare instead of the lexicographic one)
        double *s_x = reinterpret_cast<double *>(s_p);
        for (int k = threadIdx.x; k < len; k += ST_THREADS) s_x[k] = (k < cnt) ? cand[k].x : INFINITY;
        __syncthreads();
        for (int k = 2; k <= len; k <<= 1) {
            for (int j = k >> 1; j > 0; j >>= 1) {
                for (int i = threadIdx.x; i < len; i += ST_THREADS) {
                    const int ixj = i ^ j;
                    if (ixj > i) {
                        const double a = s_x[i], b = s_x[ixj];
                        const bool up = ((i & k) == 0);
                        if ((a > b) == up) { s_x[i] = b; s_x[ixj] = a; }
                    }
                }
                __syncthreads();
            }
        }
        for (int q = threadIdx.x; q < 2 * B; q += ST_THREADS) {
            const int b = q >> 1, k = q & 1;
            if (P.xm_slot[b][k] == s) P.xm_val[b][k] = s_x[P.xm_rank[b][k]];
        }
        return;
    }
    for (int k = threadIdx.x; k < len; k += ST_THREADS) s_p[k] = (k < cnt) ? cand[k] : make_double2(INFINITY, INFINITY);
    __syncthreads();
    for (int k = 2; k <= len; k <<= 1) {
        for (int j = k >> 1; j > 0; j >>= 1) {
            for (int i = threadIdx.x; i < len; i += ST_THREADS) {
                const int ixj = i ^ j;
                if (ixj > i) {
                    const double2 a = s_p[i], b = s_p[ixj];
                    const bool up = ((i & k) == 0);
                    if (pair_gt(a, b) == up) { s_p[i] = b; s_p[ixj] = a; }
                }
            }
            __syncthreads();
        }
    }
    // x medians living in this slot
    for (int q = threadIdx.x; q < 2 * B; q += ST_THREADS) {
        const int b = q >> 1, k = q & 1;
        if (P.xm_slot[b][k] == s) P.xm_val[b][k] = s_p[P.xm_rank[b][k]].x;
    }
    if (P.slot_boundary[s]) {
        // exact bin of every pair from its rank; their variances join the bins' histograms; keep them sorted for T6
        int *g = T.yhist + (size_t)row * MAXB * NBY;
        const long long pre = P.slot_prefix[s];
        for (int k = threadIdx.x; k < cnt; k += ST_THREADS) {
            const double2 pr = s_p[k];
            cand[k] = pr;
            atomicAdd(&g[bin_of_rank(pre + k, n, B) * NBY + ybucket(pr.y, P.yb0, T.geom)], 1);
        }
    }
}

// a CTA walks the slots blockIdx.x, blockIdx.x + gridDim.x, ... of its row: almost all of them were settled by k_xselect,
// so a thin grid keeps the (usually empty) launches cheap
template <int THREADS, int CAP_LO, int CAP_HI>
__global__ void __launch_bounds__(THREADS, (THREADS == 256) ? 4 : (CAP_HI <= 4096 ? 2 : 1)) k_xresolve(TrendBuffers T, long long n, int B, int nslot_max)
{
    extern __shared__ double2 s_p[];
    __shared__ int s_skip;                       // the row's fallback flag, read once for the whole CTA (other CTAs may set it meanwhile)
    if (threadIdx.x == 0) s_skip = T.plan[blockIdx.y].fallback;
    __syncthreads();
    if (s_skip) return;
    for (int s = blockIdx.x; s < nslot_max; s += gridDim.x) {
        xresolve_slot<THREADS, CAP_LO, CAP_HI>(T, n, B, blockIdx.y, s, s_p);
        __syncthreads();
    }
}

// ------------------------------------------------------------------ T5
__global__ void __launch_bounds__(256) k_yplan(TrendBuffers T, long long n, int B)
{
    __shared__ int s_pre[NBY + 1];
    const long long row = blockIdx.y;
    const int b = blockIdx.x;
    RowPlan &P = T.plan[row];
    if (P.fallback) return;
    const long long lo = ((long long)b * n) / B, hi = ((long long)(b + 1) * n) / B;
    const long long w = hi - lo;
    if (w <= 0) return;
    const int *h = T.yhist + ((size_t)row * MAXB + b) * NBY;
    {   // exclusive prefix over the NBY buckets: four per thread, warp scan, eight warp totals
        static_assert(NBY == 4 * 256, "k_yplan: four buckets per thread");
        __shared__ int s_wsum[8];
        const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
        const int4 v = reinterpret_cast<const int4 *>(h)[threadIdx.x];
        const int mine = v.x + v.y + v.z + v.w;
        int inc = mine;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) { const int o = __shfl_up_sync(0xffffffffu, inc, d); if (lane >= d) inc += o; }
        if (lane == 31) s_wsum[wid] = inc;
        __syncthreads();
        int base = inc - mine;
        for (int q = 0; q < wid; ++q) base += s_wsum[q];
        s_pre[4 * threadIdx.x + 0] = base; s_pre[4 * threadIdx.x + 1] = base + v.x;
        s_pre[4 * threadIdx.x + 2] = base + v.x + v.y; s_pre[4 * threadIdx.x + 3] = base + v.x + v.y + v.z;
        if (threadIdx.x == 255) s_pre[NBY] = base + mine;
        __syncthreads();
    }
    if (threadIdx.x == 0) {
        const int acc = s_pre[NBY];
        if (acc != (int)w) { atomicOr(&P.fallback, FB_YTOTAL); }
        else {
            auto bucket_of = [&](long long r) {
                int l = 0, hgh = NBY;
                while (hgh - l > 1) { const int mid = (l + hgh) >> 1; if ((long long)s_pre[mid] <= r) l = mid; else hgh = mid; }
                return l;
            };
            const long long r1 = w / 2;
            const int b1 = bucket_of(r1);
            P.ym_bucket[b][1] = b1; P.ym_rank[b][1] = (int)(r1 - s_pre[b1]); P.ym_count[b][1] = s_pre[b1 + 1] - s_pre[b1];
            P.ym_bucket[b][0] = -1; P.ym_count[b][0] = 0;
            if ((w & 1) == 0) {
                const long long r0 = r1 - 1;
                const int b0 = bucket_of(r0);
                P.ym_bucket[b][0] = b0; P.ym_rank[b][0] = (int)(r0 - s_pre[b0]); P.ym_count[b][0] = s_pre[b0 + 1] - s_pre[b0];
            }
        }
    }
}

// ------------------------------------------------------------------ T6
__device__ __forceinline__ void ycollect_append(TrendBuffers &T, long long row, int bin, int k, double y)
{
    const size_t slot = ((size_t)row * MAXB + bin) * 2 + k;
    const int pos = atomicAdd(&T.ycand_cnt[slot], 1);
    if (pos < T.capy) T.ycand[slot * T.capy + pos] = y;
    else {                                                   // massive ties (variances on their floor): remember the range
        const unsigned long long key = (unsigned long long)__double_as_longlong(y);
        atomicMin(&T.yover_min[slot], key);
        atomicMax(&T.yover_max[slot], key);
    }
}

// the variance belongs to slot 1 (upper median bucket) or 0 (lower median bucket, when it is a different bucket) of its bin
__device__ __forceinline__ void ycollect_one(TrendBuffers &T, long long row, const int2 *s_yb, int bin, double y, int yb0)
{
    const int yb = ybucket(y, yb0, T.geom);
    const int2 t = s_yb[bin];
    if (yb == t.y) ycollect_append(T, row, bin, 1, y);
    else if (yb == t.x) ycollect_append(T, row, bin, 0, y);
}

__global__ void __launch_bounds__(ST_THREADS) k_ycollect(const double *__restrict__ V, long long n, long long row_stride, TrendBuffers T, int B)
{
    // T3 left (bin, variance bucket) of every pair as a 16-bit code: this pass reads those two bytes per pair, eight pairs per
    // 128-bit load, and fetches the variance itself only for the ~2 % that sit in a bin's median bucket(s)
    constexpr int YQ_CAP = 8192;                         // matches queued per 131072-pair chunk (typically ~2600)
    static_assert(CHUNK <= (1 << 17), "queue entries keep the offset inside the chunk in 17 bits");
    __shared__ int2 s_yb[MAXB];
    __shared__ long long s_lo[MAXB];
    __shared__ unsigned s_q[YQ_CAP];
    __shared__ int s_qn;
    __shared__ int s_cnt[2 * MAXB], s_base[2 * MAXB];
    extern __shared__ unsigned char s_hit[];             // [32768] per code: 0 = not wanted, 1 + k = the bin's median bucket k
    const long long row = blockIdx.y;
    const RowPlan &P = T.plan[row];
    if (P.fallback) return;
    for (int k = threadIdx.x; k < MAXB; k += ST_THREADS) s_yb[k] = k < B ? make_int2(P.ym_bucket[k][0], P.ym_bucket[k][1]) : make_int2(-1, -1);
    for (int k = threadIdx.x; k < 32768 / 16; k += ST_THREADS) reinterpret_cast<uint4 *>(s_hit)[k] = make_uint4(0u, 0u, 0u, 0u);
    if (threadIdx.x == 0) s_qn = 0;
    if (threadIdx.x < 2 * MAXB) s_cnt[threadIdx.x] = 0;
    __syncthreads();
    if (threadIdx.x < 2 * B) {                           // (k = 0 first: when both medians share a bucket it is filed as k = 1)
        const int bin = threadIdx.x >> 1, k = threadIdx.x & 1;
        const int yb = k ? s_yb[bin].y : s_yb[bin].x;
        if (yb >= 0 && yb < NBY && !(k == 0 && yb == s_yb[bin].y)) s_hit[(bin << 10) | yb] = (unsigned char)(1 + k);
    }
    __syncthreads();
    const long long c0 = (long long)blockIdx.x * CHUNK, c1 = min(n, c0 + CHUNK);
    const double *v = V + row * row_stride;
    const unsigned short *codes = T.codes + row * T.code_stride;
    constexpr int YU = 4;                                // 128-bit loads in flight per thread
    for (long long jb0 = c0 + 8LL * threadIdx.x; jb0 < c1; jb0 += 8LL * ST_THREADS * YU) {
        uint4 qs[YU];
#pragma unroll
        for (int r = 0; r < YU; ++r) {
            const long long jb = jb0 + 8LL * ST_THREADS * r;
            qs[r] = jb < c1 ? *reinterpret_cast<const uint4 *>(codes + jb) : make_uint4(~0u, ~0u, ~0u, ~0u);
        }
#pragma unroll
        for (int r = 0; r < YU; ++r) {
            const long long jb = jb0 + 8LL * ST_THREADS * r;
            const unsigned w[4] = {qs[r].x, qs[r].y, qs[r].z, qs[r].w};
            const int valid = (int)min(8LL, c1 - jb);    // (<= 0 for the all-ones filler; < 8 only at the end of the row)
#pragma unroll
            for (int u = 0; u < 8; ++u) {
                const unsigned code = (w[u >> 1] >> (16 * (u & 1))) & 0xFFFFu;
                const unsigned hit = code < 0x8000u ? s_hit[code] : 0u;
                if (hit && u < valid) {
                    // ~2 % of the pairs.  A global atomic round trip here would stall the warp once per match: matches are
                    // queued in shared memory (target << 17 | offset in the chunk) and filed by the whole CTA afterwards
                    // (a ballot-aggregated push was measured slower)
                    const int bin = (int)(code >> 10), k = (int)hit - 1;
                    const int qp = atomicAdd(&s_qn, 1);
                    if (qp < YQ_CAP) { s_q[qp] = ((unsigned)(bin * 2 + k) << 17) | (unsigned)(jb + u - c0); atomicAdd(&s_cnt[bin * 2 + k], 1); }
                    else ycollect_append(T, row, bin, k, v[jb + u]);
                }
            }
        }
    }
    __syncthreads();
    const int qn = min(s_qn, YQ_CAP);
    // one global atomic per (CTA, slot) reserves the slot's range for this chunk's matches -- every CTA of a row bumping the
    // same 2B counters once per match was what this pass spent its time on -- and the matches take consecutive places in it
    if (threadIdx.x < 2 * MAXB) {
        const int c = s_cnt[threadIdx.x];
        s_base[threadIdx.x] = c ? atomicAdd(&T.ycand_cnt[(size_t)row * MAXB * 2 + threadIdx.x], c) : 0;
        s_cnt[threadIdx.x] = 0;
    }
    __syncthreads();
    for (int i = threadIdx.x; i < qn; i += ST_THREADS) {
        const unsigned e = s_q[i];
        const int tgt = (int)(e >> 17);
        const double y = v[c0 + (e & 0x1FFFFu)];
        const int pos = s_base[tgt] + atomicAdd(&s_cnt[tgt], 1);
        const size_t slot = (size_t)row * MAXB * 2 + tgt;
        if (pos < T.capy) T.ycand[slot * T.capy + pos] = y;
        else {                                                   // massive ties (variances on their floor): remember the range
            const unsigned long long key = (unsigned long long)__double_as_longlong(y);
            atomicMin(&T.yover_min[slot], key);
            atomicMax(&T.yover_max[slot], key);
        }
    }
    // the partitioned / sorted boundary slots of T4 (their pairs carry no code): shared out over the row's CTAs; the bin of
    // rank r is the number of bin boundaries floor(b n / B), b >= 1, at or below r
    for (int b = threadIdx.x; b < B; b += ST_THREADS) s_lo[b] = ((long long)b * n) / B;
    __syncthreads();
    for (int sl = blockIdx.x; sl < P.nslot; sl += gridDim.x) {
        if (!P.slot_boundary[sl]) continue;
        const double2 *cand = T.cand + ((size_t)row * MAXSLOT + sl) * CAPX;
        const long long pre = P.slot_prefix[sl];
        int bin0 = 0;
        while (bin0 + 1 < B && s_lo[bin0 + 1] <= pre) ++bin0;
        for (int k = threadIdx.x; k < P.slot_count[sl]; k += ST_THREADS) {
            int bin = bin0;
            while (bin + 1 < B && s_lo[bin + 1] <= pre + k) ++bin;
            ycollect_one(T, row, s_yb, bin, cand[k].y, P.yb0);
        }
    }
}

// ------------------------------------------------------------------ T7

__device__ void yresolve_bin(TrendBuffers &T, long long n, int B, long long row, int b, double *s_v)
{
    // sort the collected variances of the bin's target bucket(s), pick the median rank(s)
    __shared__ int s_fail;
    RowPlan &P = T.plan[row];
    if (P.ybin_done[b]) return;
    const long long lo = ((long long)b * n) / B, hi = ((long long)(b + 1) * n) / B;
    if (hi <= lo) return;
    if (threadIdx.x == 0) s_fail = 0;
    __syncthreads();
    double ym[2] = {0.0, 0.0};
    for (int k = 0; k < 2; ++k) {
        if (P.ym_bucket[b][k] < 0) continue;
        if (k == 0 && P.ym_bucket[b][0] == P.ym_bucket[b][1]) continue;       // same bucket: resolved with k = 1
        const int cnt = T.ycand_cnt[(row * MAXB + b) * 2 + k];
        if (cnt != P.ym_count[b][k]) { if (threadIdx.x == 0) s_fail = FB_YCOUNT; }
        else if (cnt > T.capy) { if (threadIdx.x == 0) s_fail = FB_YSLOT; }
        __syncthreads();
        if (s_fail) break;
        int len = 1;
        while (len < cnt) len <<= 1;
        const double *src = T.ycand + (((size_t)row * MAXB + b) * 2 + k) * T.capy;
        for (int q = threadIdx.x; q < len; q += 256) s_v[q] = q < cnt ? src[q] : INFINITY;
        __syncthreads();
        for (int kk = 2; kk <= len; kk <<= 1)
            for (int j = kk >> 1; j > 0; j >>= 1) {
                for (int i = threadIdx.x; i < len; i += 256) {
                    const int ixj = i ^ j;
                    if (ixj > i) {
                        const double a = s_v[i], c = s_v[ixj];
                        const bool up = ((i & kk) == 0);
                        if ((a > c) == up) { s_v[i] = c; s_v[ixj] = a; }
                    }
                }
                __syncthreads();
            }
        ym[k] = s_v[P.ym_rank[b][k]];
        if (k == 1 && P.ym_bucket[b][0] == P.ym_bucket[b][1]) ym[0] = s_v[P.ym_rank[b][0]];
        __syncthreads();
    }
    if (threadIdx.x == 0) {
        if (s_fail) atomicOr(&P.fallback, s_fail);
        else { P.ym_val[b][0] = ym[0]; P.ym_val[b][1] = ym[1]; }
    }
}

// (bins blockIdx.x, blockIdx.x + gridDim.x, ... of row blockIdx.y: k_yselect leaves almost nothing, so the grid is thin)
__global__ void __launch_bounds__(256) k_yresolve(TrendBuffers T, long long n, int B)
{
    extern __shared__ double s_v[];              // capy
    __shared__ int s_skip;
    if (threadIdx.x == 0) s_skip = T.plan[blockIdx.y].fallback;
    __syncthreads();
    if (s_skip) return;
    for (int b = blockIdx.x; b < B; b += gridDim.x) {
        yresolve_bin(T, n, B, blockIdx.y, b, s_v);
        __syncthreads();
    }
}

__device__ void knots_from_bins(const double *bx, const double *by, const double *bw, int used, Knots *out);

__global__ void k_row_knots(TrendBuffers T, long long n, int B, Knots *knots, int *row_fallback)
{
    const long long row = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (row >= T.rows) return;
    const RowPlan &P = T.plan[row];
    if (P.fallback) { row_fallback[row] = P.fallback; return; }
    double bx[MAXB], by[MAXB], bw[MAXB];
    int used = 0;
    for (int b = 0; b < B; ++b) {
        const long long lo = ((long long)b * n) / B, hi = ((long long)(b + 1) * n) / B;
        const long long w = hi - lo;
        if (w <= 0) continue;
        bx[used] = (w & 1) ? P.xm_val[b][1] : 0.5 * (P.xm_val[b][0] + P.xm_val[b][1]);
        by[used] = (w & 1) ? P.ym_val[b][1] : 0.5 * (P.ym_val[b][0] + P.ym_val[b][1]);
        bw[used] = (double)w;
        ++used;
    }
    row_fallback[row] = 0;
    knots_from_bins(bx, by, bw, used, knots + row);
}

// bin medians -> PAVA -> de-duplicated knots (wls_backend.c:507-560, 262-338)
__device__ void knots_from_bins(const double *bx, const double *by, const double *bw, int used, Knots *out)
{
    Knots K;
    K.nk = 0; K.constant = 0; K.cval = 1.0e-8;
    if (used == 1) { K.constant = 1; K.cval = fmax(by[0], 1.0e-8); *out = K; return; }
    double pv[MAX_KNOTS], pw[MAX_KNOTS], fit[MAX_KNOTS];
    int pl[MAX_KNOTS], nb = 0;
    for (int i = 0; i < used; ++i) {
        pv[nb] = by[i]; pw[nb] = fmax(bw[i], 1.0e-8); pl[nb] = 1; ++nb;
        while (nb >= 2 && pv[nb - 2] > pv[nb - 1]) {
            const double tw = __dadd_rn(pw[nb - 2], pw[nb - 1]);
            const double mv = __dadd_rn(__dmul_rn(pv[nb - 2], pw[nb - 2]), __dmul_rn(pv[nb - 1], pw[nb - 1])) / tw;
            pv[nb - 2] = mv; pw[nb - 2] = tw; pl[nb - 2] += pl[nb - 1];
            --nb;
        }
    }
    int q = 0;
    for (int b = 0; b < nb; ++b) for (int r = 0; r < pl[b]; ++r) fit[q++] = pv[b];
    int nk = 0;
    for (int b = 0; b < used; ++b) {
        const double cx = bx[b], cy = fmax(fit[b], 1.0e-8);
        if (nk > 0 && cx <= K.x[nk - 1]) { K.y[nk - 1] = fmax(K.y[nk - 1], cy); continue; }
        K.x[nk] = cx; K.y[nk] = cy; ++nk;
    }
    K.nk = nk;
    if (nk == 1) { K.constant = 1; K.cval = fmax(K.y[0], 1.0e-8); }
    *out = K;
}

__global__ void k_knots_serial(const double *bx, const double *by, const double *bw, int used, Knots *out)
{
    if (threadIdx.x == 0 && blockIdx.x == 0) knots_from_bins(bx, by, bw, used, out);
}

// ------------------------------------------------------------------ host driver
int trend_knots_select(const double *d_C, double *d_V, long long m, long long n, long long row_stride, Knots *d_knots,
                       int *d_row_fallback, int fused_window, cudaStream_t st)
{
    // fused_window > 0: V is not computed yet -- the first pass produces it together with the |C| histogram and T3's
    // 32-bit key of every pair
    const int B = (int)fmax(4.0, floor(1.0 + (log((double)n + 1.0) / log(2.0))));      // wls_backend.c:456
    if (B > MAXB) return ST_INVALID;
    Arena ar(st);
    TrendBuffers T{};
    T.rows = m;
    T.geom = bucket_geometry(n);
    T.capy = CAPY_MAX;          // 16384 variances per (bin, median) slot: 8 MB per row of scratch
    RB_TRY(ar.alloc(&T.xhist, (size_t)m * NBX));
    RB_TRY(ar.alloc(&T.lut, (size_t)m * NBX));
    RB_TRY(ar.alloc(&T.binlo, (size_t)m * NBX));
    RB_TRY(ar.alloc(&T.plan, (size_t)m));
    RB_TRY(ar.alloc(&T.cand, (size_t)m * MAXSLOT * CAPX));
    RB_TRY(ar.alloc(&T.cand_cnt, (size_t)m * MAXSLOT));
    RB_TRY(ar.alloc(&T.yhist, (size_t)m * MAXB * NBY));
    RB_TRY(ar.alloc(&T.ycand, (size_t)m * MAXB * 2 * T.capy));
    RB_TRY(ar.alloc(&T.ycand_cnt, (size_t)m * MAXB * 2));
    T.code_stride = (n + 7) & ~7LL;
    RB_TRY(ar.alloc(&T.codes, (size_t)m * (size_t)T.code_stride));
    if (fused_window > 0) RB_TRY(ar.alloc(&T.keys, (size_t)m * (size_t)T.code_stride));
    RB_CUDA(cudaMemsetAsync(T.xhist, 0, sizeof(int) * (size_t)m * NBX, st));
    RB_CUDA(cudaMemsetAsync(T.cand_cnt, 0, sizeof(int) * (size_t)m * MAXSLOT, st));
    RB_CUDA(cudaMemsetAsync(T.yhist, 0, sizeof(int) * (size_t)m * MAXB * NBY, st));
    RB_CUDA(cudaMemsetAsync(T.ycand_cnt, 0, sizeof(int) * (size_t)m * MAXB * 2, st));
    RB_TRY(ar.alloc(&T.yover_min, (size_t)m * MAXB * 2));
    RB_TRY(ar.alloc(&T.yover_max, (size_t)m * MAXB * 2));
    RB_CUDA(cudaMemsetAsync(T.yover_min, 0xFF, sizeof(unsigned long long) * (size_t)m * MAXB * 2, st));
    RB_CUDA(cudaMemsetAsync(T.yover_max, 0, sizeof(unsigned long long) * (size_t)m * MAXB * 2, st));

    static bool attr_dev[64] = {false};
    int attr_d = 0;
    cudaGetDevice(&attr_d);
    bool &attr = attr_dev[attr_d & 63];
    const size_t sm_xhist = sizeof(int) * NBX;
    const size_t sm_collect = sizeof(int) * (size_t)B * NBY + 2 * NBX;      // histograms + the 16-bit bucket table
    const size_t sm_resolve = sizeof(double2) * CAPX;
    const size_t sm_plan = sizeof(int) * (NBX + 258) + sizeof(double) * YSAMPLE + sizeof(SelScratch);
    if (!attr) {
        RB_CUDA(cudaFuncSetAttribute(k_xhist, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm_xhist));
        RB_CUDA(cudaFuncSetAttribute(k_ycollect, cudaFuncAttributeMaxDynamicSharedMemorySize, 32768));
        RB_CUDA(cudaFuncSetAttribute(k_xcollect, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(sizeof(int) * MAXB * NBY + 2 * NBX)));
        RB_CUDA(cudaFuncSetAttribute(k_xcollect_keys, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(sizeof(int) * MAXB * NBY + 2 * NBX)));
        RB_CUDA(cudaFuncSetAttribute(k_xresolve<512, 4096, CAPX>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm_resolve));
        RB_CUDA(cudaFuncSetAttribute(k_xresolve<512, 2048, 4096>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(sizeof(double2) * 4096)));
        RB_CUDA(cudaFuncSetAttribute(k_xplan, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm_plan));
        RB_CUDA(cudaFuncSetAttribute(k_yresolve, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(sizeof(double) * CAPY_MAX)));
        RB_CUDA(cudaFuncSetAttribute(k_xselect<512, 2048, CAPX>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(sizeof(unsigned long long) * 2 * CAPX)));
        RB_CUDA(cudaFuncSetAttribute(k_yselect<256, 4096, CAPY_MAX>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(sizeof(unsigned long long) * CAPY_MAX)));
        attr = true;
    }
    const unsigned chunks = (unsigned)((n + CHUNK - 1) / CHUNK);
    const dim3 gstream(chunks, (unsigned)m);
    if (fused_window > 0) {
        const size_t sm_fused = sizeof(int) * NBX / 2 + 2 * sizeof(double) * rv_buf(fused_window);
        static bool attr2_dev[64] = {false};
    int attr2_d = 0;
    cudaGetDevice(&attr2_d);
    bool &attr2 = attr2_dev[attr2_d & 63];
        if (!attr2) {
            const int mx = (int)(sizeof(int) * NBX / 2 + 2 * sizeof(double) * rv_buf(RV_MAXW));
            RB_CUDA(cudaFuncSetAttribute(k_rollvar_xhist<31>, cudaFuncAttributeMaxDynamicSharedMemorySize, mx));
            RB_CUDA(cudaFuncSetAttribute(k_rollvar_xhist<0>, cudaFuncAttributeMaxDynamicSharedMemorySize, mx));
            attr2 = true;
        }
        RB_PROF("k_rollvar_xhist", st, (double)m * n * 20.0);
        const dim3 grv((unsigned)((n + RV_CHUNK - 1) / RV_CHUNK), (unsigned)m);
        if (fused_window == 31)
            k_rollvar_xhist<31><<<grv, RV_THREADS, sm_fused, st>>>(d_C, n, row_stride, fused_window, d_V, T.xhist, T.geom, T.keys, T.code_stride);
        else
            k_rollvar_xhist<0><<<grv, RV_THREADS, sm_fused, st>>>(d_C, n, row_stride, fused_window, d_V, T.xhist, T.geom, T.keys, T.code_stride);
        RB_LAUNCH_CHECK();
    } else {
        RB_PROF("trend_xhist", st, (double)m * n * 8.0);
        k_xhist<<<gstream, ST_THREADS, sm_xhist, st>>>(d_C, n, row_stride, T.xhist, T.geom);
        RB_LAUNCH_CHECK();
    }
    {
        RB_PROF("trend_plan_resolve", st, 0.0);
        k_xplan<<<(unsigned)m, 256, sm_plan, st>>>(T, d_V, row_stride, n, B);
        RB_LAUNCH_CHECK();
    }
    {
        // fused pass: 4 B of keys + 2 B of codes per pair (the gathers of slot pairs are not counted); else C, V and codes
        RB_PROF("trend_xcollect", st, (double)m * n * (T.keys ? 6.0 : 18.0));
        if (T.keys) k_xcollect_keys<<<(unsigned)sm_count(), XC_THREADS, sm_collect, st>>>(d_C, d_V, n, row_stride, T, B);
        else k_xcollect<<<(unsigned)sm_count(), XC_THREADS, sm_collect, st>>>(d_C, d_V, n, row_stride, T, B);
        RB_LAUNCH_CHECK();
    }
    {
        RB_PROF("trend_plan_resolve", st, 0.0);
        const unsigned nslot_max = (unsigned)std::min(MAXSLOT, 3 * B);
        // selection first (one or two ranks per slot, or one boundary to partition around); the sort kernels then only see
        // what it left: short rows whose buckets span several bins
        k_xselect<256, -1, 2048><<<dim3(nslot_max, (unsigned)m), 256, sizeof(unsigned long long) * 2 * 2048, st>>>(T, n, B);
        RB_LAUNCH_CHECK();
        k_xselect<512, 2048, CAPX><<<dim3(nslot_max, (unsigned)m), 512, sizeof(unsigned long long) * 2 * CAPX, st>>>(T, n, B);
        RB_LAUNCH_CHECK();
        k_xresolve<256, -1, 2048><<<dim3(std::min(nslot_max, 8u), (unsigned)m), 256, sizeof(double2) * 2048, st>>>(T, n, B, (int)nslot_max);
        RB_LAUNCH_CHECK();
        k_xresolve<512, 2048, 4096><<<dim3(std::min(nslot_max, 8u), (unsigned)m), 512, sizeof(double2) * 4096, st>>>(T, n, B, (int)nslot_max);
        RB_LAUNCH_CHECK();
        k_xresolve<512, 4096, CAPX><<<dim3(std::min(nslot_max, 8u), (unsigned)m), 512, sm_resolve, st>>>(T, n, B, (int)nslot_max);
        RB_LAUNCH_CHECK();
        k_yplan<<<dim3((unsigned)B, (unsigned)m), 256, 0, st>>>(T, n, B);
        RB_LAUNCH_CHECK();
    }
    {
        RB_PROF("trend_ycollect", st, (double)m * n * 2.0);
        k_ycollect<<<gstream, ST_THREADS, 32768, st>>>(d_V, n, row_stride, T, B);
        RB_LAUNCH_CHECK();
    }
    {
        RB_PROF("trend_plan_resolve", st, 0.0);
        k_yselect<256, -1, 4096><<<dim3((unsigned)B, (unsigned)m), 256, sizeof(unsigned long long) * 4096, st>>>(T, n, B);
        RB_LAUNCH_CHECK();
        k_yselect<256, 4096, CAPY_MAX><<<dim3((unsigned)B, (unsigned)m), 256, sizeof(unsigned long long) * T.capy, st>>>(T, n, B);
        RB_LAUNCH_CHECK();
        k_yresolve<<<dim3((unsigned)std::min(B, 4), (unsigned)m), 256, sizeof(double) * T.capy, st>>>(T, n, B);
        RB_LAUNCH_CHECK();
        k_row_knots<<<(unsigned)((m + 63) / 64), 64, 0, st>>>(T, n, B, d_knots, d_row_fallback);
        RB_LAUNCH_CHECK();
    }
    return 0;
}

}  // namespace score
}  // namespace rb
