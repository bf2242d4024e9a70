// Cross-fit Whittaker baseline as overlapped tiles of a parallel second-order recurrence.
//
// Replaces /root/reference/rocco/native/baseline_backend.c:79-303 (per row, per parity: a
// pentadiagonal LDL^T factorisation and three sequential substitution sweeps of length n).
//
// What makes it parallel:
//  * the factor of  W_p + lambda D'D  depends only on (n, lambda, parity); past the first few hundred
//    rows it sits on a period-2 steady state (to ~1e-12, the conditioning noise of the recurrence
//    itself) and only the last two rows deviate.  The host computes a short head table, the steady
//    pair and a 4-entry tail once per (n, lambda);
//  * forward / backward substitution are second-order linear recurrences, i.e. IIR filters whose
//    impulse response decays like rho^k, rho = 0.9775 for the default window (lambda(101) = 4.67e5).  Each tile is
//    solved with a halo of HALO bins on both sides from a zero state; the truncation error at the tile is
//    0.9775^1280 ~ 2e-13 of the signal, below the reference's own ~1e-10 noise floor;
//  * rho grows with lambda (1 - rho ~ 0.59 lambda^-1/4): 0.9849 at window 151, 0.9977 at window 1001, where rho^1280 is
//    5e-2.  build_factor computes rho from the steady pair and admits the tiles only while rho^HALO and rho^1536 (the
//    streaming kernel's truncated cross-warp sum) are <= WT_TILE_TAU = 1e-12: windows up to 105 (lambda <= 5.5e5).
//    Above that, rows longer than the head table take k_whittaker_exact, which replays the reference's sequential solve
//    operation for operation (the same bits as baseline_backend.c), one thread per (row, parity);
//  * every thread owns ITEMS consecutive bins: a zero-state local sweep, a scan of the 2-vector
//    carry across threads, then the true sweep.  Both parities run interleaved in the same thread
//    (two independent dependency chains).
//
// Kernels:
//  * k_whittaker_stream: interior ("steady") tiles, whose coefficients are the period-2 steady state.  A
//    persistent grid of two-CTA clusters, one cluster per tile region at a time;
//  * k_whittaker: the first and last tile(s) of a row, which read the head and tail tables, and every tile at penalties
//    below ~10 (WP_REDERIVE_GROWTH_MAX).  One CTA per region, with a general carry scan over per-chunk transitions;
//  * k_small_rows: rows shorter than 25 bins;
//  * k_whittaker_exact + k_whittaker_exact_out: penalties the tiles cannot carry (above).
//
// Both tile kernels fuse the reference's Python prologue: y = log2(max(x,0)+1) - pilot_row
// (inference.py:40-47, 333-334) and the epilogue  centered = y - baseline  (inference.py:338).
#include "common.cuh"
#include "score.cuh"

#include <cooperative_groups.h>
#include <math.h>

#include <algorithm>
#include <atomic>
#include <map>
#include <memory>
#include <mutex>

namespace rb {
namespace score {

constexpr int WT_REGION = 12288;                   // bins solved per CTA
constexpr int WT_HALO = 1280;
constexpr int WT_OUT = WT_REGION - 2 * WT_HALO;    // 9728 bins written per CTA
constexpr int WT_THREADS_G = 512, WT_ITEMS_G = 24; // edge tiles (k_whittaker): one CTA per region
constexpr int HEAD_LEN = 4096;
// Largest decay rho^k, over the shortest distance k a truncated state is carried in the tile kernels, at which they are
// used.  A tile's truncation error is at most about rho^k max|y| (measured in a float64 emulation of one steady tile at
// windows 151 to 1001: 0.1 to 0.25 rho^1280 max|y|).  The reference's own float64 solve is off by ~1e-11 max|y| already
// at the default penalty, and by more above it, so 1e-12 keeps the truncation an order of magnitude under that error:
// the kernels stay as accurate as the reference wherever they are used.
constexpr double WT_TILE_TAU = 1e-12;
// The streaming kernel re-derives the forward solution right to left over a thread's WP_GEOM_ITEMS bins, which multiplies
// its rounding by r^-WP_GEOM_ITEMS, r the smaller per-bin root modulus of the forward recurrence: 1.3 at the default
// penalty, but 2e3 at window 3 and 1e18 at lambda = 1e-3.  Up to 64 (r >= 0.71, lambda >~ 10) that stays below 1e-14
// of the signal; smaller penalties send the interior tiles to k_whittaker, which stores the forward solution instead.
constexpr double WP_REDERIVE_GROWTH_MAX = 64.0;

// ------------------------------------------------------------------ host: factor tables
static void host_factor(long long n_true, long long len, int parity, double lam,
                        std::vector<double> &d, std::vector<double> &l1, std::vector<double> &l2)
{
    // Same recurrences and association order as baseline_backend.c:106-140.  `n_true` decides which rows
    // carry the end bands; only the first `len` rows are produced.
    auto a0 = [&](long long i) {
        const double w = ((i & 1) == parity) ? 1.0 : 0.0;
        if (i == 0 || i == n_true - 1) return w + lam;
        if (i == 1 || i == n_true - 2) return w + (5.0 * lam);
        return w + (6.0 * lam);
    };
    auto a1 = [&](long long i) { return (i == 0 || i == n_true - 2) ? (-2.0 * lam) : (-4.0 * lam); };
    d.assign(len, 0.0); l1.assign(len, 0.0); l2.assign(len, 0.0);
    double t1, t2;
    d[0] = a0(0);
    if (len == 1) return;
    l1[0] = a1(0) / d[0];
    l2[0] = lam / d[0];
    d[1] = a0(1) - ((l1[0] * l1[0]) * d[0]);
    if (n_true > 2) { t1 = ((l2[0] * d[0]) * l1[0]); l1[1] = (a1(1) - t1) / d[1]; }
    if (n_true > 3) l2[1] = lam / d[1];
    for (long long i = 2; i < len; ++i) {
        t1 = ((l1[i - 1] * l1[i - 1]) * d[i - 1]);
        t2 = ((l2[i - 2] * l2[i - 2]) * d[i - 2]);
        d[i] = a0(i) - t1 - t2;
        if (i <= n_true - 2) { t1 = ((l2[i - 1] * d[i - 1]) * l1[i - 1]); l1[i] = (a1(i) - t1) / d[i]; }
        if (i <= n_true - 3) l2[i] = lam / d[i];
    }
}

// Tables of the streaming kernel for one alignment shift parity `ap` (region position 0 has index parity ap):
// chain A carries the rhs of the even region positions (parity p = ap), chain B the odd ones (p = 1 - ap).
constexpr int WP_HALF = 6144;                      // bins per CTA, two CTAs per region
constexpr int WP_MAXWARPS = 16;
constexpr int WP_LEVELS = 9;                       // 5 in-warp levels + 4 across the warps of a CTA
// thread geometry of the streaming kernel (threads x bins per thread = WP_HALF): 512 x 12 (384 x 16 and a cluster of four
// 256-thread CTAs were measured slower: fewer resident warps / no gain from the finer phases)
constexpr int WP_GEOM_THREADS = 512, WP_GEOM_ITEMS = 12;
constexpr int WP_CROSS_WARP_BINS = 4 * 32 * WP_GEOM_ITEMS;   // span of the streaming kernel's truncated cross-warp sum
struct PairTab {
    double cf[2][3][2];                            // [chain][dinv, l1, l2][position parity]
    double trans[2][2][WP_LEVELS][4];              // [chain][fwd/bwd][level]: transition over ITEMS * 2^level bins
    double g[2][16][2];                            // [chain][j]: response of the zero-state backward sweep of a chunk to z_j = 1: (x_0, x_1)
    double il2[2][2];                              // [chain][position parity]: 1 / l2 (the forward recurrence run right to left)
};
struct PairPow {
    double lane[2][2][2][32][2];                   // [chain][dir][matrix row][k]: row of T^k chunks (k = 0: identity); 16-byte lane stride
    double warp[2][2][WP_MAXWARPS][4];             // [chain][dir][w]: T^(32 w) chunks (w = 0: identity)
};

struct FactorHost {
    int head_len = 0;
    PairTab pair_tab[2];                           // [alignment shift parity]
    PairPow pair_pow[2];
    std::vector<double> head[2][3];      // [parity][dinv,l1,l2][head_len]
    double steady[2][3][2];              // [parity][coef][index parity]
    double tail[2][3][4];                // rows n-4 .. n-1
    double decay[2] = {0.0, 0.0};        // [parity]: rho, the per-bin decay of the steady recurrence
    bool tiles_exact = true;             // rho^WT_HALO and rho^WP_CROSS_WARP_BINS <= WT_TILE_TAU (always for short rows)
    bool stream_stable = true;           // r^-WP_GEOM_ITEMS <= WP_REDERIVE_GROWTH_MAX (see above)
};

static void mat2_mul(const double *a, const double *b, double *c)   // c = a*b (row-major 2x2)
{
    double r[4] = {a[0] * b[0] + a[1] * b[2], a[0] * b[1] + a[1] * b[3], a[2] * b[0] + a[3] * b[2], a[2] * b[1] + a[3] * b[3]};
    for (int k = 0; k < 4; ++k) c[k] = r[k];
}

static void build_factor(long long n, double lam, FactorHost &F)
{
    const bool small = n <= HEAD_LEN + 8;
    const long long len = small ? n : HEAD_LEN;
    F.head_len = (int)len;
    for (int p = 0; p < 2; ++p) {
        std::vector<double> d, l1, l2;
        host_factor(n, len, p, lam, d, l1, l2);
        F.head[p][0].resize(len); F.head[p][1] = l1; F.head[p][2] = l2;
        for (long long i = 0; i < len; ++i) F.head[p][0][i] = 1.0 / d[i];
        for (int q = 0; q < 2; ++q) {       // placeholders for short rows (every tile takes the general path)
            const long long idx = std::min<long long>(len - 1, std::max<long long>(0, len - 2 + q));
            F.steady[p][0][q] = F.head[p][0][idx]; F.steady[p][1][q] = l1[idx]; F.steady[p][2][q] = l2[idx];
        }
        if (!small) {
            // steady state by index parity (len is even here), then the four end rows continued from it
            for (int q = 0; q < 2; ++q) {
                F.steady[p][0][q] = 1.0 / d[len - 2 + q]; F.steady[p][1][q] = l1[len - 2 + q]; F.steady[p][2][q] = l2[len - 2 + q];
            }
            double dd[6], e1[6], e2[6];         // rows n-6 .. n-1; first two from the steady state
            for (int k = 0; k < 2; ++k) {
                const long long i = n - 6 + k;
                dd[k] = d[len - 2 + (i & 1)]; e1[k] = l1[len - 2 + (i & 1)]; e2[k] = l2[len - 2 + (i & 1)];
            }
            for (int k = 2; k < 6; ++k) {
                const long long i = n - 6 + k;
                const double w = ((i & 1) == p) ? 1.0 : 0.0;
                const double m0 = (i == n - 1) ? w + lam : (i == n - 2) ? w + (5.0 * lam) : w + (6.0 * lam);
                const double m1 = (i == n - 2) ? (-2.0 * lam) : (-4.0 * lam);
                double t1 = ((e1[k - 1] * e1[k - 1]) * dd[k - 1]);
                double t2 = ((e2[k - 2] * e2[k - 2]) * dd[k - 2]);
                dd[k] = m0 - t1 - t2;
                e1[k] = 0.0; e2[k] = 0.0;
                if (i <= n - 2) { t1 = ((e2[k - 1] * dd[k - 1]) * e1[k - 1]); e1[k] = (m1 - t1) / dd[k]; }
                if (i <= n - 3) e2[k] = lam / dd[k];
                F.tail[p][0][k - 2] = 1.0 / dd[k]; F.tail[p][1][k - 2] = e1[k]; F.tail[p][2][k - 2] = e2[k];
            }
            // decay per bin: square root of the spectral radius of the two-step companion matrix of the forward
            // recurrence f_i = r_i - l1[i-1] f_{i-1} - l2[i-2] f_{i-2} (the backward one is its transpose)
            const double Se[4] = {-l1[len - 1], -l2[len - 2], 1.0, 0.0};       // step onto an even index
            const double So[4] = {-l1[len - 2], -l2[len - 1], 1.0, 0.0};       // step onto an odd index
            double M[4];
            mat2_mul(So, Se, M);
            const double tr = M[0] + M[3], det = M[0] * M[3] - M[1] * M[2], disc = tr * tr - 4.0 * det;
            const double radius = disc < 0.0 ? sqrt(det) : 0.5 * (fabs(tr) + sqrt(disc));
            F.decay[p] = sqrt(radius);
            const double rmin = sqrt(fabs(det) / radius);                   // smaller per-bin root modulus
            F.stream_stable = F.stream_stable && pow(rmin, -WP_GEOM_ITEMS) <= WP_REDERIVE_GROWTH_MAX;
        } else {
            for (int k = 0; k < 4; ++k) F.tail[p][0][k] = F.tail[p][1][k] = F.tail[p][2][k] = 0.0;
        }
    }
    // (a NaN decay, from lambda = 0 or not finite, fails the test too)
    for (int p = 0; p < 2 && !small; ++p)
        F.tiles_exact = F.tiles_exact && pow(F.decay[p], WT_HALO) <= WT_TILE_TAU && pow(F.decay[p], WP_CROSS_WARP_BINS) <= WT_TILE_TAU;
    // streaming kernel: chains by region-position parity, for both alignment shift parities
    constexpr int WP_ITEMS = WP_GEOM_ITEMS, WP_WARPS = WP_GEOM_THREADS / 32;
    for (int ap = 0; ap < 2; ++ap) {
        PairTab &T = F.pair_tab[ap];
        PairPow &W = F.pair_pow[ap];
        for (int ch = 0; ch < 2; ++ch) {
            const int p = ch ^ ap;                                  // parity mask served by this chain
            for (int k = 0; k < 3; ++k)
                for (int q = 0; q < 2; ++q) T.cf[ch][k][q] = F.steady[p][k][q ^ ap];
            for (int q = 0; q < 2; ++q) T.il2[ch][q] = 1.0 / T.cf[ch][2][q];
            double Tf[4] = {1, 0, 0, 1}, Tb[4] = {1, 0, 0, 1};
            for (int j = 0; j < WP_ITEMS; ++j) {                    // position j of a chunk (chunks start on even positions)
                const double S[4] = {-T.cf[ch][1][(j + 1) & 1], -T.cf[ch][2][j & 1], 1.0, 0.0};
                mat2_mul(S, Tf, Tf);
            }
            for (int j = WP_ITEMS - 1; j >= 0; --j) {
                const double S[4] = {-T.cf[ch][1][j & 1], -T.cf[ch][2][j & 1], 1.0, 0.0};
                mat2_mul(S, Tb, Tb);
            }
            for (int k = 0; k < 4; ++k) { T.trans[ch][0][0][k] = Tf[k]; T.trans[ch][1][0][k] = Tb[k]; }
            for (int j0 = 0; j0 < 16; ++j0) {
                double a1 = 0.0, a2 = 0.0;
                for (int j = WP_ITEMS - 1; j >= 0 && j0 < WP_ITEMS; --j) {
                    const double na = (j == j0 ? 1.0 : 0.0) - T.cf[ch][2][j & 1] * a2 - T.cf[ch][1][j & 1] * a1;
                    a2 = a1; a1 = na;
                }
                T.g[ch][j0][0] = a1; T.g[ch][j0][1] = a2;
            }
            for (int dct = 0; dct < 2; ++dct) {
                for (int l = 1; l < WP_LEVELS; ++l) mat2_mul(T.trans[ch][dct][l - 1], T.trans[ch][dct][l - 1], T.trans[ch][dct][l]);
                double acc[4] = {1, 0, 0, 1};
                for (int k = 0; k < 32; ++k) {
                    for (int q = 0; q < 4; ++q) W.lane[ch][dct][q >> 1][k][q & 1] = acc[q];
                    mat2_mul(T.trans[ch][dct][0], acc, acc);
                }
                double wacc[4] = {1, 0, 0, 1};
                for (int w = 0; w < WP_WARPS; ++w) {
                    for (int q = 0; q < 4; ++q) W.warp[ch][dct][w][q] = wacc[q];
                    mat2_mul(T.trans[ch][dct][5], wacc, wacc);
                }
            }
        }
    }
}

// ------------------------------------------------------------------ fast log2 for arguments >= 1
// v = 2^e * m, m in [1,2); i = top 7 mantissa bits; r = m * inv[i] - 1 with inv[i] ~ 1/(1 + (i + 0.5)/128), |r| <= 2^-8;
// log2(v) = e + (tab[i] + log2(1 + r)), tab[i] = -log2(inv[i]) for the ROUNDED inv[i], log2(1+r) by a degree-7 polynomial
// (truncation < 2^-66).  Total error ~1 ulp of the result for v >= 2 and < 3e-19 absolute near 1: four orders of
// magnitude below the solver's own noise floor, at ~25 issue slots instead of ~110 for the library log2.
struct Log2Tables { double inv[128]; double tab[128]; };
static Log2Tables g_log2_host;
static bool g_log2_ready = false;

static void build_log2_tables()
{
    if (g_log2_ready) return;
    for (int i = 0; i < 128; ++i) {
        const long double c = 1.0L + ((long double)i + 0.5L) / 128.0L;
        const double inv = (double)(1.0L / c);
        g_log2_host.inv[i] = inv;
        g_log2_host.tab[i] = (double)(-log2l((long double)inv));
    }
    g_log2_ready = true;
}

// polynomial coefficients live in the constant bank: a DFMA reads them as an operand, whereas 64-bit immediates cost two
// uniform moves each per use
__constant__ double c_log2poly[7] = {
    0.20609929155656704,      //  1/(7 ln2)
    -0.24044917348266152,     // -1/(6 ln2)
    0.28853900817779268,      //  1/(5 ln2)
    -0.36067376022224085,     // -1/(4 ln2)
    0.48089834696298783,      //  1/(3 ln2)
    -0.72134752044448170,     // -1/(2 ln2)
    1.4426950408889634,       //  1/ln2
};

__device__ __forceinline__ double fast_log2_ge1(double v, const double *s_inv, const double *s_tab)
{
    const long long bits = __double_as_longlong(v);
    const long long mant = bits & 0x000FFFFFFFFFFFFFLL;
    const int e = (int)(bits >> 52) - 1023;
    const int i = (int)(mant >> 45);
    const double m = __longlong_as_double(mant | 0x3FF0000000000000LL);
    const double r = __fma_rn(m, s_inv[i], -1.0);
    // log2(1+r) = r/ln2 * (1 - r/2 + r^2/3 - ...)
    double p = c_log2poly[0];
#pragma unroll
    for (int k = 1; k < 7; ++k) p = __fma_rn(p, r, c_log2poly[k]);
    const double res = (double)e + __fma_rn(p, r, s_tab[i]);
    return mant == 0 ? (double)e : res;                              // exact powers of two (zero counts -> 0.0), branch-free
}


// Leaner variant for the streaming kernel: a 32-entry interleaved table {inv[i], tab[i]} (one 128-bit shared load; 512 bytes, so
// that the 32 lanes' lookups rarely collide on a bank), |r| <= 2^-6 and the degree-7 polynomial above (truncation
// r^8 / (8 ln 2) < 1e-15 absolute, five orders below the solver's noise floor), exponent converted with the 2^52 trick
// instead of I2F.  Exact for powers of two (zero counts give 0.0) like the function above.
constexpr int LOG2_V2_ENTRIES = 34;               // centres 1 + i/32, i = 0..32 (+1 pad: the bulk copy moves multiples of 16 bytes anyway)
__device__ __forceinline__ double fast_log2_ge1_v2(double v, const double2 *s_it)
{
    const int hi = __double2hiint(v), lo = __double2loint(v);
    const int mhi = hi & 0x000FFFFF;
    const double2 it = s_it[(mhi + 0x4000) >> 15];           // nearest centre; entry 0 is {1, 0}: m = 1 gives r = 0 and log2 = e exactly
    const double m = __hiloint2double(mhi | 0x3FF00000, lo);
    const double r = __fma_rn(m, it.x, -1.0);
    double p = c_log2poly[0];
#pragma unroll
    for (int k = 1; k < 7; ++k) p = __fma_rn(p, r, c_log2poly[k]);
    // exponent as a double: 2^52 + (biased exponent) - (2^52 + 1023)
    const double e = __hiloint2double(0x43300000, hi >> 20) - 4503599627371519.0;
    return e + __fma_rn(p, r, it.y);
}

// ------------------------------------------------------------------ device side
struct WhitParams {
    const void *x;              // input matrix rows (f64 or f32) or already-transformed rows
    const double *pilot;        // per-row offset subtracted after the log transform (nullptr: none)
    double *out;                // centered (mode 0) or baseline (mode 1), row-major like x
    int *bad;                   // set to 1 when a non-finite input/result is seen
    const double *head[2][3];   // device head tables
    double steady[2][3][2];
    double tail[2][3][4];
    const double *log2tab;      // device copy of Log2Tables (inv[128], tab[128])
    long long n;
    long long row_stride;       // elements between rows of x / out
    int head_len;
    int rows;
    int tiles_per_row;
    int tile_offset;            // this launch covers tiles [tile_offset, tile_offset + span_tiles) of every row
    int span_tiles;
    int in_f32;                 // 1: x is float32
    int log_transform;          // 1: y = log2(max(x,0)+1) - pilot ; 0: y = x
    int write_baseline;         // 1: out = baseline ; 0: out = y - baseline
};

__device__ __forceinline__ double load_y(const WhitParams &P, long long row, long long i, const double *s_log = nullptr)
{
    double v = P.in_f32 ? (double)reinterpret_cast<const float *>(P.x)[row * P.row_stride + i]
                        : reinterpret_cast<const double *>(P.x)[row * P.row_stride + i];
    if (P.log_transform) {
        if (!isfinite(v)) return NAN;            // inference.py:45-46 rejects non-finite input (fmax would swallow NaN / -inf)
        v = fmax(v, 0.0) + 1.0;
        v = s_log ? fast_log2_ge1(v, s_log, s_log + 128) : log2(v);
        if (P.pilot) v -= P.pilot[row];
    }
    return v;
}

__device__ __forceinline__ double coef(const WhitParams &P, int p, int k, long long i)
{
    if (i < P.head_len) return P.head[p][k][i];
    if (i >= P.n - 4) return P.tail[p][k][i - (P.n - 4)];
    return P.steady[p][k][i & 1];
}

// General carry scan (chunks with their own transition matrices: first / last tile of a row).
template <int THREADS>
__device__ __forceinline__ void carry_scan_general(double &v0, double &v1, double m00, double m01, double m10, double m11,
                                                   bool reverse, double *s_buf /* [6 * THREADS] */)
{
    constexpr int WT_THREADS = THREADS;
    // plain Hillis-Steele in shared memory over (M, v) affine maps; x -> M x + v
    const int t = threadIdx.x;
    const int pos = reverse ? WT_THREADS - 1 - t : t;
    double *sm = s_buf;
    auto put = [&](int p) {
        sm[p * 6 + 0] = m00; sm[p * 6 + 1] = m01; sm[p * 6 + 2] = m10; sm[p * 6 + 3] = m11;
        sm[p * 6 + 4] = v0; sm[p * 6 + 5] = v1;
    };
    put(pos);
    __syncthreads();
    for (int d = 1; d < WT_THREADS; d <<= 1) {
        double o[6];
        const bool act = pos >= d;
        if (act) for (int k = 0; k < 6; ++k) o[k] = sm[(pos - d) * 6 + k];
        __syncthreads();
        if (act) {
            // new = me o older :  M = Mme*Mold ; v = Mme*vold + vme
            const double nv0 = m00 * o[4] + m01 * o[5] + v0, nv1 = m10 * o[4] + m11 * o[5] + v1;
            const double n00 = m00 * o[0] + m01 * o[2], n01 = m00 * o[1] + m01 * o[3];
            const double n10 = m10 * o[0] + m11 * o[2], n11 = m10 * o[1] + m11 * o[3];
            m00 = n00; m01 = n01; m10 = n10; m11 = n11; v0 = nv0; v1 = nv1;
            put(pos);
        }
        __syncthreads();
    }
}

// First and last tile(s) of a row: the coefficients vary along the region (head table, tail rows, row ends) and the
// region may be short, so every chunk builds its own transition and the carry scan is the general one.
template <int WT_THREADS, int WT_ITEMS>
__global__ void __launch_bounds__(WT_THREADS, 1) k_whittaker(WhitParams P)
{
    constexpr int WT_PAD = WT_ITEMS + 1;
    extern __shared__ double smem[];
    double *s_f0 = smem;                             // WT_THREADS * WT_PAD
    double *s_f1 = smem + WT_THREADS * WT_PAD;
    __shared__ double s_log[256];                     // fast-log2 tables: inv[128], tab[128]
    for (int k = threadIdx.x; k < 256; k += WT_THREADS) s_log[k] = P.log2tab[k];
    __syncthreads();

    const int tid = threadIdx.x;
    const long long row = blockIdx.x / P.span_tiles;
    const int tile = P.tile_offset + blockIdx.x % P.span_tiles;
    const long long out0 = (long long)tile * WT_OUT;                 // first bin written by this CTA
    const long long out1 = min(P.n, out0 + WT_OUT);
    long long r0 = out0 - WT_HALO; if (r0 < 0) r0 = 0;               // region solved (even start)
    long long r1 = out1 + WT_HALO; if (r1 > P.n) r1 = P.n;
    const int rlen = (int)(r1 - r0);

    // ---- stage rhs (masked y) for both parities, coalesced; four loads in flight per thread before any arithmetic
    int bad = 0;
    const bool keep_y = !P.write_baseline;
    const int o_lo = (int)(out0 - r0), o_hi = (int)(out1 - r0);            // region positions of the tile's own bins
    const long long rbase = row * P.row_stride + r0;
    const float *xf = reinterpret_cast<const float *>(P.x) + rbase;
    const double *xd = reinterpret_cast<const double *>(P.x) + rbase;
    double *outp = P.out + rbase;
    const double pil = (P.log_transform && P.pilot) ? P.pilot[row] : 0.0;
    const bool par0 = ((r0 & 1) == 0);
    constexpr int LD = 4;
#pragma unroll 1
    for (int e0 = tid; e0 < WT_REGION; e0 += LD * WT_THREADS) {
        double raw[LD];
#pragma unroll
        for (int u = 0; u < LD; ++u) {
            const int e = e0 + u * WT_THREADS;
            raw[u] = (e < rlen) ? (P.in_f32 ? (double)xf[e] : xd[e]) : 0.0;
        }
#pragma unroll
        for (int u = 0; u < LD; ++u) {
            const int e = e0 + u * WT_THREADS;
            if (e >= WT_REGION) break;
            double y = 0.0;
            if (e < rlen) {
                y = raw[u];
                // inference.py:45-46 rejects non-finite input (fmax would swallow NaN / -inf); a finite input gives a
                // finite y, so one test serves both the input check and the result check
                const bool fin = isfinite(y);
                if (P.log_transform) y = fin ? fast_log2_ge1(fmax(y, 0.0) + 1.0, s_log, s_log + 128) - pil : NAN;
                bad |= !fin;
                // park y of the tile's own bins in the output buffer: the epilogue needs it again and a second
                // log2 per bin costs more issue slots than an L2 round trip
                if (keep_y && e >= o_lo && e < o_hi) outp[e] = y;
            }
            const int a = e + e / WT_ITEMS;
            const bool even = (((e & 1) == 0) == par0);
            s_f0[a] = even ? y : 0.0;
            s_f1[a] = even ? 0.0 : y;
        }
    }
    if (bad) *P.bad = 1;
    __syncthreads();

    const int base = tid * WT_ITEMS;                                  // first region position of this thread
    const long long i0 = r0 + base;                                   // global index of that bin
    double *f0 = s_f0 + tid * WT_PAD, *f1 = s_f1 + tid * WT_PAD;
    const int cnt = max(0, min(WT_ITEMS, rlen - base));
    double *s_buf = reinterpret_cast<double *>(smem + 2 * WT_THREADS * WT_PAD);

    // ================= forward substitution  L f = rhs
    // pass A: zero-state sweep -> end vector (f[last], f[last-1]) and the chunk transition
    double e00 = 0.0, e01 = 0.0, e10 = 0.0, e11 = 0.0;        // parity0: (f, fprev) ; parity1: (f, fprev)
    double ha[2][4];                                          // homogeneous solutions per parity
    for (int p = 0; p < 2; ++p) { ha[p][0] = 1.0; ha[p][1] = 0.0; ha[p][2] = 0.0; ha[p][3] = 1.0; }
    {
        double a1 = 0.0, a2 = 0.0, b1 = 0.0, b2 = 0.0;        // f[i-1], f[i-2] per parity
#pragma unroll
        for (int j = 0; j < WT_ITEMS; ++j) {
            if (j < cnt) {
                const long long i = i0 + j;
                const double l1a = i >= 1 ? coef(P, 0, 1, i - 1) : 0.0, l2a = i >= 2 ? coef(P, 0, 2, i - 2) : 0.0;
                const double l1b = i >= 1 ? coef(P, 1, 1, i - 1) : 0.0, l2b = i >= 2 ? coef(P, 1, 2, i - 2) : 0.0;
                // homogeneous: h[i] = -l1 h[i-1] - l2 h[i-2] for the two unit start states
                for (int p = 0; p < 2; ++p) {
                    const double l1 = p ? l1b : l1a, l2 = p ? l2b : l2a;
                    const double n0 = -l1 * ha[p][0] - l2 * ha[p][2], n1 = -l1 * ha[p][1] - l2 * ha[p][3];
                    ha[p][2] = ha[p][0]; ha[p][3] = ha[p][1]; ha[p][0] = n0; ha[p][1] = n1;
                }
                const double na = fma(-l2a, a2, fma(-l1a, a1, f0[j]));
                const double nb = fma(-l2b, b2, fma(-l1b, b1, f1[j]));
                a2 = a1; a1 = na; b2 = b1; b1 = nb;
            }
        }
        e00 = a1; e01 = a2; e10 = b1; e11 = b2;
    }
    // carry: state entering chunk t = inclusive scan value of chunk t-1
    double in00, in01, in10, in11;
    carry_scan_general<WT_THREADS>(e00, e01, ha[0][0], ha[0][1], ha[0][2], ha[0][3], false, s_buf);
    carry_scan_general<WT_THREADS>(e10, e11, ha[1][0], ha[1][1], ha[1][2], ha[1][3], false, s_buf);
    in00 = __shfl_up_sync(0xffffffffu, e00, 1); in01 = __shfl_up_sync(0xffffffffu, e01, 1);
    in10 = __shfl_up_sync(0xffffffffu, e10, 1); in11 = __shfl_up_sync(0xffffffffu, e11, 1);
    {
        __shared__ double s_edge[WT_THREADS / 32][4];
        if ((tid & 31) == 31) { s_edge[tid >> 5][0] = e00; s_edge[tid >> 5][1] = e01; s_edge[tid >> 5][2] = e10; s_edge[tid >> 5][3] = e11; }
        __syncthreads();
        if ((tid & 31) == 0) {
            if (tid == 0) { in00 = in01 = in10 = in11 = 0.0; }
            else { const int w = (tid >> 5) - 1; in00 = s_edge[w][0]; in01 = s_edge[w][1]; in10 = s_edge[w][2]; in11 = s_edge[w][3]; }
        }
        __syncthreads();
    }
    // pass B: true sweep, scaled by 1/d on the way out (z = f / d)
    {
        double a1 = in00, a2 = in01, b1 = in10, b2 = in11;
#pragma unroll
        for (int j = 0; j < WT_ITEMS; ++j) {
            if (j < cnt) {
                const long long i = i0 + j;
                const double l1a = i >= 1 ? coef(P, 0, 1, i - 1) : 0.0, l2a = i >= 2 ? coef(P, 0, 2, i - 2) : 0.0;
                const double l1b = i >= 1 ? coef(P, 1, 1, i - 1) : 0.0, l2b = i >= 2 ? coef(P, 1, 2, i - 2) : 0.0;
                const double da = coef(P, 0, 0, i), db = coef(P, 1, 0, i);
                const double na = fma(-l2a, a2, fma(-l1a, a1, f0[j]));
                const double nb = fma(-l2b, b2, fma(-l1b, b1, f1[j]));
                a2 = a1; a1 = na; b2 = b1; b1 = nb;
                f0[j] = na * da; f1[j] = nb * db;
            }
        }
    }

    // ================= backward substitution  L' x = z   (right to left)
    for (int p = 0; p < 2; ++p) { ha[p][0] = 1.0; ha[p][1] = 0.0; ha[p][2] = 0.0; ha[p][3] = 1.0; }
    {
        double a1 = 0.0, a2 = 0.0, b1 = 0.0, b2 = 0.0;        // x[i+1], x[i+2]
#pragma unroll
        for (int j = WT_ITEMS - 1; j >= 0; --j) {
            if (j < cnt) {
                const long long i = i0 + j;
                const double l1a = (i + 1 < P.n) ? coef(P, 0, 1, i) : 0.0, l2a = (i + 2 < P.n) ? coef(P, 0, 2, i) : 0.0;
                const double l1b = (i + 1 < P.n) ? coef(P, 1, 1, i) : 0.0, l2b = (i + 2 < P.n) ? coef(P, 1, 2, i) : 0.0;
                for (int p = 0; p < 2; ++p) {
                    const double l1 = p ? l1b : l1a, l2 = p ? l2b : l2a;
                    const double n0 = -l1 * ha[p][0] - l2 * ha[p][2], n1 = -l1 * ha[p][1] - l2 * ha[p][3];
                    ha[p][2] = ha[p][0]; ha[p][3] = ha[p][1]; ha[p][0] = n0; ha[p][1] = n1;
                }
                const double na = fma(-l2a, a2, fma(-l1a, a1, f0[j]));
                const double nb = fma(-l2b, b2, fma(-l1b, b1, f1[j]));
                a2 = a1; a1 = na; b2 = b1; b1 = nb;
            }
        }
        e00 = a1; e01 = a2; e10 = b1; e11 = b2;
    }
    carry_scan_general<WT_THREADS>(e00, e01, ha[0][0], ha[0][1], ha[0][2], ha[0][3], true, s_buf);
    carry_scan_general<WT_THREADS>(e10, e11, ha[1][0], ha[1][1], ha[1][2], ha[1][3], true, s_buf);
    in00 = __shfl_down_sync(0xffffffffu, e00, 1); in01 = __shfl_down_sync(0xffffffffu, e01, 1);
    in10 = __shfl_down_sync(0xffffffffu, e10, 1); in11 = __shfl_down_sync(0xffffffffu, e11, 1);
    {
        __shared__ double s_edge2[WT_THREADS / 32][4];
        if ((tid & 31) == 0) { s_edge2[tid >> 5][0] = e00; s_edge2[tid >> 5][1] = e01; s_edge2[tid >> 5][2] = e10; s_edge2[tid >> 5][3] = e11; }
        __syncthreads();
        if ((tid & 31) == 31) {
            if (tid == WT_THREADS - 1) { in00 = in01 = in10 = in11 = 0.0; }
            else { const int w = (tid >> 5) + 1; in00 = s_edge2[w][0]; in01 = s_edge2[w][1]; in10 = s_edge2[w][2]; in11 = s_edge2[w][3]; }
        }
        __syncthreads();
    }
    {
        double a1 = in00, a2 = in01, b1 = in10, b2 = in11;
#pragma unroll
        for (int j = WT_ITEMS - 1; j >= 0; --j) {
            if (j < cnt) {
                const long long i = i0 + j;
                const double l1a = (i + 1 < P.n) ? coef(P, 0, 1, i) : 0.0, l2a = (i + 2 < P.n) ? coef(P, 0, 2, i) : 0.0;
                const double l1b = (i + 1 < P.n) ? coef(P, 1, 1, i) : 0.0, l2b = (i + 2 < P.n) ? coef(P, 1, 2, i) : 0.0;
                const double na = fma(-l2a, a2, fma(-l1a, a1, f0[j]));
                const double nb = fma(-l2b, b2, fma(-l1b, b1, f1[j]));
                a2 = a1; a1 = na; b2 = b1; b1 = nb;
                f0[j] = 0.5 * (na + nb);                       // cross-fit average (baseline_backend.c:296-299)
            }
        }
    }
    __syncthreads();

    // ---- write the tile (coalesced); y comes back from where the staging loop parked it (an L2 hit)
    int bad2 = 0;
    constexpr int LDE = 4;
#pragma unroll 1
    for (int e0 = o_lo + tid; e0 < o_hi; e0 += LDE * WT_THREADS) {
        double yv[LDE];
#pragma unroll
        for (int u = 0; u < LDE; ++u) {
            const int e = e0 + u * WT_THREADS;
            yv[u] = (!P.write_baseline && e < o_hi) ? __ldcg(outp + e) : 0.0;
        }
#pragma unroll
        for (int u = 0; u < LDE; ++u) {
            const int e = e0 + u * WT_THREADS;
            if (e >= o_hi) break;
            const double b = s_f0[e + e / WT_ITEMS];
            const double v = P.write_baseline ? b : yv[u] - b;
            bad2 |= !isfinite(v);
            outp[e] = v;
        }
    }
    if (bad2) *P.bad = 1;
}


// ------------------------------------------------------------------ steady tiles: streaming cluster-pair kernel
// A 12288-bin region (9728 own bins + two 1280-bin halos) is solved by a CLUSTER of two CTAs, each holding one half
// (6144 bins), and two CTAs are resident per SM, so that the barrier-separated phases of one overlap the sweeps of the
// other.  The grid is PERSISTENT: as many clusters as are co-resident walk the (row, tile) list, and the raw input of a
// cluster's next tile is in flight (bulk async copy, cp.async.bulk completing on an mbarrier, into the second of two
// landing buffers) while the current one is solved, so that neither the load latency at the start of a tile nor the
// drain of its bulk store at the end is exposed; the scan tables are loaded once per CTA.
//   * every thread reads its own consecutive bins with 128-bit shared loads and keeps y = log2(max(x,0)+1) - pilot in
//     registers;
//   * the carry scan runs inside the warp (shuffles), across the warps, and across the two CTAs: the left CTA hands its
//     total to the right one for the forward substitution, the right CTA to the left one for the backward substitution,
//     with st.async into the peer's shared memory (DSMEM) completing on the peer's mbarrier -- only the receiver waits,
//     and there is no cluster-scope fence after start-up (which would also invalidate L1);
//   * the true forward sweep also accumulates the zero-state end vector of the chunk's backward sweep, which is linear
//     in the z_j (table g), so the backward substitution needs one sweep instead of two;
//   * the forward solution is not stored: the backward sweep re-derives it by running the forward recurrence right to
//     left from the chunk's final state (n_{j-2} = (r_j - n_j - l1 n_{j-1}) / l2; twelve steps of a recurrence whose
//     reverse growth is 1/0.9775 per bin, i.e. ~1e-16 relative);
//   * the result is written over the thread's own slots of the landing buffer and leaves from there as ONE bulk store
//     per CTA (whole lines; a scalar head/tail element where the row start is only 8-byte aligned).
// A bulk copy needs a 16-byte aligned source: the region starts `shift` bins left of the tile's nominal (even) start.
// An odd shift swaps which parity mask sits on the even region positions, hence the per-launch chain tables.
struct PairParams {
    const void *x; const double *pilot; double *out; int *bad;
    const double *pow_tab;      // PairPow of this shift parity (device)
    const double *log2tab;      // LOG2_V2_ENTRIES x {inv, tab} interleaved (device)
    PairTab tab;
    long long n, row_stride;
    int row0, row_step;         // rows handled by this launch: row0 + k * row_step
    int tile_offset, span_tiles;
    int shift;
    int log_transform, write_baseline;
    int total_pairs;            // (row, tile) pairs of this launch
    double w_y, w_b;            // output = w_b * (b_even + b_odd) + w_y * y  ((1, -0.5) centred, (0, 0.5) baseline)
};

__device__ __forceinline__ unsigned smem_u32(const void *p) { return (unsigned)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_wait(unsigned mbar, unsigned parity)
{
    unsigned done = 0;
    while (!done) {
        asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}"
                     : "=r"(done) : "r"(mbar), "r"(parity) : "memory");
    }
}
__device__ __forceinline__ void bulk_load(unsigned dst, const void *src, unsigned bytes, unsigned mbar)
{
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 ::"r"(dst), "l"(src), "r"(bytes), "r"(mbar) : "memory");
}

constexpr int WP_POW_LANE = 2 * 2 * 32 * 4;               // doubles in PairPow::lane

// Carry scan of both chains at once.  v[0..1]: chain A zero-state end vector of this thread's chunk, v[2..3]: chain B.
// On exit `in` holds the true state entering the chunk.  REV: scan runs right to left (backward substitution).
//   1. Kogge-Stone inside the warp (shuffles, T^(2^l chunks));
//   2. every warp publishes its total; the state entering a warp is the sum over the FOUR warps before it in scan order of
//      T^(32 j chunks) x total -- a transition over 128 chunks (1536 bins) is below 1e-15, so older warps do not matter --
//      formed by four lanes in parallel and summed with two butterfly shuffles (no serial section, one CTA barrier);
//   3. the warps next to the CTA boundary add the peer CTA's total, which arrives by st.async on this CTA's mbarrier.
template <int WP_WARPS>
__device__ __forceinline__ void warp_entry_state(double (&E)[4], int target, int D, bool use_peer, const double (*s_wex)[4],
                                                 const double *s_pow, const double (*s_nbr)[4])
{
    // state entering scan-order warp `target`: lane group member k-1 handles the warp k places earlier
    const int k = (threadIdx.x & 3) + 1;
    const int ws = target - k;
    double2 t0 = make_double2(0.0, 0.0), t1 = make_double2(0.0, 0.0);
    int wsel = k - 1;
    bool have = false;
    if (ws >= 0) {
        t0 = *reinterpret_cast<const double2 *>(&s_wex[ws][0]); t1 = *reinterpret_cast<const double2 *>(&s_wex[ws][2]);
        have = true;
    } else if (ws == -1 && use_peer) {            // the peer's total is the state entering scan-order warp 0
        t0 = *reinterpret_cast<const double2 *>(&s_nbr[D][0]); t1 = *reinterpret_cast<const double2 *>(&s_nbr[D][2]);
        have = true;
    }
    E[0] = E[1] = E[2] = E[3] = 0.0;
    if (have) {
        const double2 *wa = reinterpret_cast<const double2 *>(s_pow + WP_POW_LANE + ((0 * 2 + D) * WP_MAXWARPS + wsel) * 4);
        const double2 *wb = reinterpret_cast<const double2 *>(s_pow + WP_POW_LANE + ((1 * 2 + D) * WP_MAXWARPS + wsel) * 4);
        const double2 a0 = wa[0], a1 = wa[1], b0 = wb[0], b1 = wb[1];
        E[0] = fma(a0.x, t0.x, a0.y * t0.y); E[1] = fma(a1.x, t0.x, a1.y * t0.y);
        E[2] = fma(b0.x, t1.x, b0.y * t1.y); E[3] = fma(b1.x, t1.x, b1.y * t1.y);
    }
#pragma unroll
    for (int q = 0; q < 4; ++q) {
        E[q] += __shfl_xor_sync(0xffffffffu, E[q], 1);
        E[q] += __shfl_xor_sync(0xffffffffu, E[q], 2);
    }
}

template <bool REV, int WP_WARPS, int CL>
__device__ __forceinline__ void pair_scan(double (&v)[4], double (&in)[4], const PairParams &P, double (*s_wex)[4],
                                          const double *s_pow, double (*s_nbr)[4], unsigned long long *s_cbar, int rank,
                                          unsigned cpar)
{
    constexpr int D = REV ? 1 : 0;
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    const int lpos = REV ? 31 - lane : lane;
    const int wpos = REV ? WP_WARPS - 1 - wid : wid;
#pragma unroll
    for (int l = 0; l < 5; ++l) {
        const int dlt = 1 << l;
        double o[4];
#pragma unroll
        for (int k = 0; k < 4; ++k) o[k] = REV ? __shfl_down_sync(0xffffffffu, v[k], dlt) : __shfl_up_sync(0xffffffffu, v[k], dlt);
        if (lpos >= dlt) {
#pragma unroll
            for (int ch = 0; ch < 2; ++ch) {
                const double *T = P.tab.trans[ch][D][l];
                v[2 * ch + 0] = fma(T[0], o[2 * ch], fma(T[1], o[2 * ch + 1], v[2 * ch + 0]));
                v[2 * ch + 1] = fma(T[2], o[2 * ch], fma(T[3], o[2 * ch + 1], v[2 * ch + 1]));
            }
        }
    }
    double e[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        e[k] = REV ? __shfl_down_sync(0xffffffffu, v[k], 1) : __shfl_up_sync(0xffffffffu, v[k], 1);
        if (lpos == 0) e[k] = 0.0;
    }
    if (lpos == 31) {
        *reinterpret_cast<double2 *>(&s_wex[wpos][0]) = make_double2(v[0], v[1]);
        *reinterpret_cast<double2 *>(&s_wex[wpos][2]) = make_double2(v[2], v[3]);
    }
    __syncthreads();
    // scan order over the cluster's CTAs: ascending rank forward, descending backward.  A CTA's total leaves for the next
    // CTA in scan order WITHOUT the contribution of the CTA before it: a transition over a whole CTA (>= 3072 bins) is
    // below 1e-30, so the chain over more than two CTAs has no serial dependency.
    const bool sender = REV ? (rank > 0) : (rank < CL - 1);
    const bool receiver = REV ? (rank < CL - 1) : (rank > 0);
    const int dest = REV ? rank - 1 : rank + 1;
    if (sender && wpos == WP_WARPS - 1) {
        // this CTA's total = the state that would enter a warp after the last one; 32 bytes into the peer's shared memory,
        // completing on the peer's mbarrier
        double N[4];
        warp_entry_state<WP_WARPS>(N, WP_WARPS, D, false, s_wex, s_pow, s_nbr);
        if (lane == 0) {
            unsigned rdst, rbar;
            asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(rdst) : "r"(smem_u32(&s_nbr[D][0])), "r"(dest));
            asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(rbar) : "r"(smem_u32(&s_cbar[D])), "r"(dest));
            asm volatile("st.async.weak.shared::cluster.mbarrier::complete_tx::bytes.v2.f64 [%0], {%1, %2}, [%3];"
                         ::"r"(rdst), "d"(N[0]), "d"(N[1]), "r"(rbar) : "memory");
            asm volatile("st.async.weak.shared::cluster.mbarrier::complete_tx::bytes.v2.f64 [%0], {%1, %2}, [%3];"
                         ::"r"(rdst + 16), "d"(N[2]), "d"(N[3]), "r"(rbar) : "memory");
        }
    }
    const bool use_peer = receiver && wpos < 4;
    if (use_peer) mbar_wait(smem_u32(&s_cbar[D]), cpar);
    double E[4];
    warp_entry_state<WP_WARPS>(E, wpos, D, use_peer, s_wex, s_pow, s_nbr);
    {
        const double2 *lp = reinterpret_cast<const double2 *>(s_pow);
        const double2 a0 = lp[((0 * 2 + D) * 2 + 0) * 32 + lpos], a1 = lp[((0 * 2 + D) * 2 + 1) * 32 + lpos];
        const double2 b0 = lp[((1 * 2 + D) * 2 + 0) * 32 + lpos], b1 = lp[((1 * 2 + D) * 2 + 1) * 32 + lpos];
        in[0] = fma(a0.x, E[0], fma(a0.y, E[1], e[0]));
        in[1] = fma(a1.x, E[0], fma(a1.y, E[1], e[1]));
        in[2] = fma(b0.x, E[2], fma(b0.y, E[3], e[2]));
        in[3] = fma(b1.x, E[2], fma(b1.y, E[3], e[3]));
    }
}

template <bool F32, int WP_THREADS, int WP_ITEMS, int CL>
__global__ void __launch_bounds__(WP_THREADS, 1024 / WP_THREADS) k_whittaker_stream(const __grid_constant__ PairParams P)
{
    namespace cg = cooperative_groups;
    constexpr int CTA_BINS = WP_THREADS * WP_ITEMS;       // cluster of CL CTAs (launch attribute) = one 12288-bin region
    static_assert(CL * CTA_BINS == 2 * WP_HALF && WP_ITEMS % 4 == 0 && WP_ITEMS <= 16 && CTA_BINS >= 3072, "stream geometry");
    constexpr int WP_WARPS = WP_THREADS / 32;
    extern __shared__ __align__(128) double smem_pair[];
    double *s_buf0 = smem_pair, *s_buf1 = smem_pair + CTA_BINS;       // landing buffers (raw in, result out)
    double *s_pow = smem_pair + 2 * CTA_BINS;
    const double2 *s_log = reinterpret_cast<const double2 *>(s_pow + sizeof(PairPow) / sizeof(double));
    __shared__ __align__(8) unsigned long long s_full[2]; // raw input of buffer b has landed
    __shared__ __align__(8) unsigned long long s_tabbar;  // tables
    __shared__ __align__(8) unsigned long long s_cbar[2]; // carry from the peer CTA: [forward, backward]
    __shared__ __align__(16) double s_nbr[2][4];
    __shared__ __align__(16) double s_wex[2][WP_MAXWARPS][4];

    const int rank = (int)cg::this_cluster().block_rank();
    const int tid = threadIdx.x;
    const int cid = blockIdx.x / CL, ncl = gridDim.x / CL;
    const int total = P.total_pairs;
    constexpr unsigned BYTES = CTA_BINS * (F32 ? 4u : 8u);
    constexpr unsigned LOG_BYTES = 16u * LOG2_V2_ENTRIES;
    const bool recv_fwd = rank > 0, recv_bwd = rank < CL - 1;     // carries this CTA receives (from its left / right neighbour)

    // (row, first element of this CTA's part) of a tile: worked out by the thread that issues the tile's bulk load and left in
    // shared memory for the others (the load's mbarrier orders the two), so that nobody else pays the index divisions
    __shared__ long long s_meta[2][2];
    auto tile_meta = [&](int pair_idx, long long *row_out) -> long long {
        const long long row = P.row0 + (long long)(pair_idx / P.span_tiles) * P.row_step;
        const int tile = P.tile_offset + pair_idx % P.span_tiles;
        const long long r0 = (long long)tile * WT_OUT - WT_HALO - P.shift;
        *row_out = row;
        return row * P.row_stride + r0 + (long long)rank * CTA_BINS;
    };

    if (tid == 0) {
        asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(smem_u32(&s_full[0])));
        asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(smem_u32(&s_full[1])));
        asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(smem_u32(&s_tabbar)));
        asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(smem_u32(&s_cbar[0])));
        asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(smem_u32(&s_cbar[1])));
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(&s_tabbar)), "r"((unsigned)sizeof(PairPow) + LOG_BYTES) : "memory");
        bulk_load(smem_u32(s_pow), P.pow_tab, (unsigned)sizeof(PairPow), smem_u32(&s_tabbar));
        bulk_load(smem_u32(s_log), P.log2tab, LOG_BYTES, smem_u32(&s_tabbar));
        if (cid < total) {
            long long row0;
            const long long hb0 = tile_meta(cid, &row0);
            s_meta[0][0] = row0; s_meta[0][1] = hb0;
            asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(&s_full[0])), "r"(BYTES) : "memory");
            bulk_load(smem_u32(s_buf0), reinterpret_cast<const char *>(P.x) + hb0 * (F32 ? 4 : 8), BYTES, smem_u32(&s_full[0]));
        }
    }
    asm volatile("barrier.cluster.arrive.relaxed.aligned;" ::: "memory");
    asm volatile("barrier.cluster.wait.aligned;" ::: "memory");      // the peer's barriers exist (once per CTA)
    mbar_wait(smem_u32(&s_tabbar), 0);

    const double (*cfA)[2] = P.tab.cf[0];
    const double (*cfB)[2] = P.tab.cf[1];
    const int p0 = rank * CTA_BINS + tid * WP_ITEMS;
    const int o_lo = WT_HALO + P.shift, o_hi = o_lo + WT_OUT;
    const bool dead = (p0 + WP_ITEMS <= o_lo);            // left-halo threads only feed the forward scan
    const int q0 = max(o_lo, rank * CTA_BINS) - rank * CTA_BINS, q1 = min(o_hi, (rank + 1) * CTA_BINS) - rank * CTA_BINS;   // own bins in CTA positions
    int bad = 0;

#pragma unroll 1
    for (int it = 0, pair_idx = cid; pair_idx < total; ++it, pair_idx += ncl) {
        const int b = it & 1;
        double *buf = b ? s_buf1 : s_buf0;
        if (tid == 0) {        // this tile's carries (the previous phase of each barrier was completed and observed one tile ago)
            if (recv_fwd) asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], 32;" ::"r"(smem_u32(&s_cbar[0])) : "memory");
            if (recv_bwd) asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], 32;" ::"r"(smem_u32(&s_cbar[1])) : "memory");
        }
        mbar_wait(smem_u32(&s_full[b]), (unsigned)(it >> 1) & 1u);
        const long long row = s_meta[b][0];
        const double pil = (P.log_transform && P.pilot) ? P.pilot[row] : 0.0;

        // ---- this thread's bins: raw -> y (registers)
        double y[WP_ITEMS];
        if (F32) {
            const float4 *rp = reinterpret_cast<const float4 *>(buf) + tid * (WP_ITEMS / 4);
#pragma unroll
            for (int u = 0; u < WP_ITEMS / 4; ++u) {
                const float4 q = rp[u];
                y[4 * u + 0] = (double)q.x; y[4 * u + 1] = (double)q.y; y[4 * u + 2] = (double)q.z; y[4 * u + 3] = (double)q.w;
            }
        } else {
            const double2 *rp = reinterpret_cast<const double2 *>(buf) + tid * (WP_ITEMS / 2);
#pragma unroll
            for (int u = 0; u < WP_ITEMS / 2; ++u) { const double2 q = rp[u]; y[2 * u] = q.x; y[2 * u + 1] = q.y; }
        }
        int expmax = 0;                                   // inference.py:45-46: non-finite input is an error
#pragma unroll
        for (int j = 0; j < WP_ITEMS; ++j) expmax = max(expmax, __double2hiint(y[j]) & 0x7FF00000);
        bad |= (expmax == 0x7FF00000);
        if (P.log_transform) {
#pragma unroll
            for (int j = 0; j < WP_ITEMS; ++j) y[j] = fast_log2_ge1_v2(dmax(y[j], 0.0) + 1.0, s_log) - pil;
        }

        double v[4], in[4];
        // ================= forward substitution: zero-state sweep, carry scan, true sweep
        {
            double a1 = 0.0, a2 = 0.0, b1 = 0.0, b2 = 0.0;
#pragma unroll
            for (int j = 0; j < WP_ITEMS; ++j) {
                const double ra = (j & 1) ? 0.0 : y[j], rb_ = (j & 1) ? y[j] : 0.0;
                const double na = fma(-cfA[2][j & 1], a2, fma(-cfA[1][(j + 1) & 1], a1, ra));
                const double nb = fma(-cfB[2][j & 1], b2, fma(-cfB[1][(j + 1) & 1], b1, rb_));
                a2 = a1; a1 = na; b2 = b1; b1 = nb;
            }
            v[0] = a1; v[1] = a2; v[2] = b1; v[3] = b2;
        }
        pair_scan<false, WP_WARPS, CL>(v, in, P, s_wex[0], s_pow, s_nbr, s_cbar, rank, (unsigned)it & 1u);
        // (the scan's CTA barrier: every thread has its raw bins in registers, and the other buffer's previous store was
        // issued a whole tile phase ago)  -> start the next tile's input
        if (tid == 0 && pair_idx + ncl < total) {
            asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");          // the other buffer's result has left
            const unsigned fb = smem_u32(&s_full[b ^ 1]);
            long long rown;
            const long long hbn = tile_meta(pair_idx + ncl, &rown);
            s_meta[b ^ 1][0] = rown; s_meta[b ^ 1][1] = hbn;          // (read one tile ago for the last time: barriers in between)
            asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(fb), "r"(BYTES) : "memory");
            bulk_load(smem_u32(b ? s_buf0 : s_buf1), reinterpret_cast<const char *>(P.x) + hbn * (F32 ? 4 : 8), BYTES, fb);
        }
        double fa1 = 0.0, fa2 = 0.0, fb1 = 0.0, fb2 = 0.0;       // final forward state of the chunk: n_{last}, n_{last-1}
        v[0] = v[1] = v[2] = v[3] = 0.0;
        if (!dead) {
            double a1 = in[0], a2 = in[1], b1 = in[2], b2 = in[3];
#pragma unroll
            for (int j = 0; j < WP_ITEMS; ++j) {
                const double ra = (j & 1) ? 0.0 : y[j], rb_ = (j & 1) ? y[j] : 0.0;
                const double na = fma(-cfA[2][j & 1], a2, fma(-cfA[1][(j + 1) & 1], a1, ra));
                const double nb = fma(-cfB[2][j & 1], b2, fma(-cfB[1][(j + 1) & 1], b1, rb_));
                a2 = a1; a1 = na; b2 = b1; b1 = nb;
                const double za = na * cfA[0][j & 1], zb = nb * cfB[0][j & 1];
                v[0] = fma(P.tab.g[0][j][0], za, v[0]); v[1] = fma(P.tab.g[0][j][1], za, v[1]);
                v[2] = fma(P.tab.g[1][j][0], zb, v[2]); v[3] = fma(P.tab.g[1][j][1], zb, v[3]);
            }
            fa1 = a1; fa2 = a2; fb1 = b1; fb2 = b2;
        }
        // ================= backward substitution (right to left), the forward solution re-derived on the way
        pair_scan<true, WP_WARPS, CL>(v, in, P, s_wex[1], s_pow, s_nbr, s_cbar, rank, (unsigned)it & 1u);
        if (!dead) {
            double a1 = in[0], a2 = in[1], b1 = in[2], b2 = in[3];
#pragma unroll
            for (int j = WP_ITEMS - 1; j >= 0; --j) {
                const double za = fa1 * cfA[0][j & 1], zb = fb1 * cfB[0][j & 1];
                const double na = fma(-cfA[2][j & 1], a2, fma(-cfA[1][j & 1], a1, za));
                const double nb = fma(-cfB[2][j & 1], b2, fma(-cfB[1][j & 1], b1, zb));
                a2 = a1; a1 = na; b2 = b1; b1 = nb;
                if (j >= 2) {
                    const double ra = (j & 1) ? 0.0 : y[j], rb_ = (j & 1) ? y[j] : 0.0;
                    const double pa = fma(-cfA[1][(j + 1) & 1], fa2, ra - fa1) * P.tab.il2[0][j & 1];
                    const double pb = fma(-cfB[1][(j + 1) & 1], fb2, rb_ - fb1) * P.tab.il2[1][j & 1];
                    fa1 = fa2; fa2 = pa; fb1 = fb2; fb2 = pb;
                } else {
                    fa1 = fa2; fb1 = fb2;
                }
                // cross-fit average (baseline_backend.c:296-299) and the output in one fused step: 0.5 * (na + nb) is exact,
                // so fma(-0.5, na + nb, y) rounds once, like y - baseline; (w_y, w_b) = (1, -0.5) centred, (0, 0.5) baseline
                y[j] = fma(P.w_b, na + nb, P.w_y * y[j]);
            }
            if (!P.log_transform) {                       // (log2 of a finite count cannot overflow the solve)
                expmax = 0;
#pragma unroll
                for (int j = 0; j < WP_ITEMS; ++j) expmax = max(expmax, __double2hiint(y[j]) & 0x7FF00000);
                bad |= (expmax == 0x7FF00000);
            }
        }
        // ---- epilogue: results over this thread's own slots of the landing buffer, own bins out in bulk
        // (float input: other threads' raw slots overlap these double slots -- all raw reads precede the scans' barriers)
        if (!dead) {
            double2 *sp = reinterpret_cast<double2 *>(buf) + tid * (WP_ITEMS / 2);
#pragma unroll
            for (int u = 0; u < WP_ITEMS / 2; ++u) sp[u] = make_double2(y[2 * u], y[2 * u + 1]);
        }
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
        __syncthreads();
        double *outp = P.out + s_meta[b][1];
        if ((reinterpret_cast<uintptr_t>(outp) & 15) == 0) {
            if (tid == 0) {
                const int b0 = (q0 + 1) & ~1, b1 = q1 & ~1;
                if (q0 < b0) outp[q0] = buf[q0];
                if (b1 < q1) outp[b1] = buf[b1];
                if (b1 > b0) {
                    asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;"
                                 ::"l"(outp + b0), "r"(smem_u32(buf + b0)), "r"((unsigned)(b1 - b0) * 8u) : "memory");
                    asm volatile("cp.async.bulk.commit_group;" ::: "memory");
                }
            }
        } else {
            for (int q = q0 + tid; q < q1; q += WP_THREADS) outp[q] = buf[q];          // coalesced fallback
            __syncthreads();                              // before the buffer is handed to the next bulk load
        }
    }
    if (bad) *P.bad = 1;
    if (tid == 0) asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");    // shared memory must outlive the last read
}

// n < 25: the reference returns a zero baseline (baseline_backend.c:266-273) -> centered = y
__global__ void k_small_rows(WhitParams P)
{
    const long long total = (long long)P.rows * P.n;
    int bad = 0;
    for (long long g = (long long)blockIdx.x * blockDim.x + threadIdx.x; g < total; g += (long long)gridDim.x * blockDim.x) {
        const long long row = g / P.n, i = g % P.n;
        const double y = load_y(P, row, i);
        bad |= !isfinite(y);
        P.out[row * P.row_stride + i] = P.write_baseline ? 0.0 : y;
    }
    if (bad) *P.bad = 1;
}

// ------------------------------------------------------------------ exact path: the reference's sequential solve
// Penalties at which the tiles' truncation is not negligible (FactorHost::tiles_exact false).  One thread per (row, parity)
// replays baseline_backend.c:142-173 over the full factor of (n, lambda, parity), which every row of the call shares:
// the forward sweep, the division by the diagonal and the backward sweep, with the reference's roundings (no
// contraction into FMAs).  Parity 0 solves in place in its output row, parity 1 in `scratch`; k_whittaker_exact_out then
// forms the cross-fit average and the epilogue.  y is recomputed there with the same library log2, so both kernels see
// the same bits, and the baseline is the reference's bit for bit.
struct ExactFactor { const double *d[2], *l1[2], *l2[2]; };

__global__ void k_whittaker_exact(WhitParams P, ExactFactor F, double *scratch, long long row0, long long rows)
{
    const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= 2 * rows) return;
    const long long row = row0 + (t >> 1), n = P.n;
    const int p = (int)(t & 1);
    double *x = p ? scratch + (t >> 1) * n : P.out + row * P.row_stride;
    const double *d = F.d[p], *l1 = F.l1[p], *l2 = F.l2[p];
    auto rhs = [&](long long i) {                     // masked rhs (oracle_baseline.c masked_rhs): keeps the signed zeros
        const double y = load_y(P, row, i);
        const bool on = (int)(i & 1) == p;
        if (i < 2 || i + 2 >= n) return on ? y : 0.0;
        return __dmul_rn(on ? 1.0 : 0.0, y);
    };
    double f2 = rhs(0);
    double f1 = __dsub_rn(rhs(1), __dmul_rn(l1[0], f2));
    x[0] = __ddiv_rn(f2, d[0]);
    x[1] = __ddiv_rn(f1, d[1]);
#pragma unroll 4
    for (long long i = 2; i < n; ++i) {
        const double f = __dsub_rn(__dsub_rn(rhs(i), __dmul_rn(l1[i - 1], f1)), __dmul_rn(l2[i - 2], f2));
        x[i] = __ddiv_rn(f, d[i]);
        f2 = f1; f1 = f;
    }
    double b1 = x[n - 1];
    double b0 = __dsub_rn(x[n - 2], __dmul_rn(l1[n - 2], b1));
    x[n - 2] = b0;
#pragma unroll 4
    for (long long i = n - 2; i-- > 0;) {
        const double v = __dsub_rn(__dsub_rn(x[i], __dmul_rn(l1[i], b0)), __dmul_rn(l2[i], b1));
        x[i] = v; b1 = b0; b0 = v;
    }
}

__global__ void k_whittaker_exact_out(WhitParams P, const double *scratch, long long row0, long long rows)
{
    const long long total = rows * P.n;
    int bad = 0;
    for (long long g = (long long)blockIdx.x * blockDim.x + threadIdx.x; g < total; g += (long long)gridDim.x * blockDim.x) {
        const long long r = g / P.n, i = g % P.n, row = row0 + r;
        double *o = P.out + row * P.row_stride + i;
        const double b = __dmul_rn(0.5, __dadd_rn(*o, scratch[g]));         // baseline_backend.c:296-299
        const double y = load_y(P, row, i);                                  // NaN for a non-finite input
        const double v = P.write_baseline ? b : __dsub_rn(y, b);
        bad |= !isfinite(y) || !isfinite(v);
        *o = v;
    }
    if (bad) *P.bad = 1;
}

static std::atomic<long long> g_exact_rows{0};
long long whittaker_exact_rows() { return g_exact_rows.load(); }

static int whittaker_exact(const WhitParams &P, double lam, cudaStream_t st)
{
    // scratch bounded by the factor (6 n doubles) and up to 256 MB of parity-1 rows; released when this call returns
    const long long n = P.n, rows = P.rows;
    Arena ar(st);
    std::vector<double> h((size_t)6 * n);
    ExactFactor E;
    double *d_fac = nullptr, *d_scr = nullptr;
    RB_TRY(ar.alloc(&d_fac, (size_t)6 * n));
    for (int p = 0; p < 2; ++p) {
        std::vector<double> d, l1, l2;
        host_factor(n, n, p, lam, d, l1, l2);
        std::copy(d.begin(), d.end(), h.begin() + (3 * p + 0) * n);
        std::copy(l1.begin(), l1.end(), h.begin() + (3 * p + 1) * n);
        std::copy(l2.begin(), l2.end(), h.begin() + (3 * p + 2) * n);
        E.d[p] = d_fac + (3 * p + 0) * n; E.l1[p] = d_fac + (3 * p + 1) * n; E.l2[p] = d_fac + (3 * p + 2) * n;
    }
    // (pageable source: the call returns once h is staged, so h may die with this scope)
    RB_CUDA(cudaMemcpyAsync(d_fac, h.data(), sizeof(double) * h.size(), cudaMemcpyHostToDevice, st));
    const long long batch = std::max<long long>(1, std::min<long long>(rows, (256LL << 20) / (long long)sizeof(double) / n));
    RB_TRY(ar.alloc(&d_scr, (size_t)(batch * n)));
    for (long long r0 = 0; r0 < rows; r0 += batch) {
        const long long nr = std::min(batch, rows - r0);
        RB_PROF("k_whittaker_exact", st, (double)nr * n * ((P.in_f32 ? 4.0 : 8.0) + 8.0));
        k_whittaker_exact<<<(unsigned)((2 * nr + 63) / 64), 64, 0, st>>>(P, E, d_scr, r0, nr);
        RB_LAUNCH_CHECK();
        const int blocks = (int)std::min<long long>((nr * n + 255) / 256, (long long)sm_count() * 8);
        k_whittaker_exact_out<<<blocks, 256, 0, st>>>(P, d_scr, r0, nr);
        RB_LAUNCH_CHECK();
    }
    g_exact_rows.fetch_add(rows);
    return 0;
}

// ------------------------------------------------------------------ factor cache (device tables per (n, lambda))
// Entries are handed out as shared_ptr: a caller keeps its tables alive across its launches whatever the cache does
// meanwhile (eviction only drops the cache's own reference), and the device buffers are released by the destructor on
// every path, including a failed construction.
struct FactorDev {
    FactorHost host;
    double *d_head[2][3] = {{nullptr, nullptr, nullptr}, {nullptr, nullptr, nullptr}};
    double *d_log2 = nullptr;
    double *d_log2i = nullptr;                       // the same tables interleaved {inv[i], tab[i]} (streaming kernel)
    double *d_pairpow[2] = {};                       // PairPow per shift parity
    int device = 0;
    unsigned long long last_use = 0;
    FactorDev() = default;
    FactorDev(const FactorDev &) = delete;
    FactorDev &operator=(const FactorDev &) = delete;
    ~FactorDev()
    {
        for (int p = 0; p < 2; ++p) {
            for (int k = 0; k < 3; ++k) if (d_head[p][k]) cudaFree(d_head[p][k]);
            if (d_pairpow[p]) cudaFree(d_pairpow[p]);
        }
        if (d_log2) cudaFree(d_log2);
        if (d_log2i) cudaFree(d_log2i);
    }
};
using FactorRef = std::shared_ptr<FactorDev>;
static std::mutex g_fmutex;
static std::map<std::pair<long long, double>, FactorRef> g_fcache[16];
static unsigned long long g_fclock = 0;
constexpr size_t FACTOR_CACHE_MAX = 256;

static int upload_factor(FactorDev &F)
{
    for (int p = 0; p < 2; ++p)
        for (int k = 0; k < 3; ++k) {
            RB_CUDA(cudaMalloc(&F.d_head[p][k], sizeof(double) * std::max(1, F.host.head_len)));
            RB_CUDA(cudaMemcpy(F.d_head[p][k], F.host.head[p][k].data(), sizeof(double) * F.host.head_len, cudaMemcpyHostToDevice));
        }
    build_log2_tables();
    RB_CUDA(cudaMalloc(&F.d_log2, sizeof(Log2Tables)));
    RB_CUDA(cudaMemcpy(F.d_log2, &g_log2_host, sizeof(Log2Tables), cudaMemcpyHostToDevice));
    {
        double il[2 * LOG2_V2_ENTRIES];
        for (int i = 0; i < LOG2_V2_ENTRIES; ++i) {
            const long double c = 1.0L + (long double)i / 32.0L;
            const double inv = (double)(1.0L / c);
            il[2 * i] = inv;
            il[2 * i + 1] = (i == 0) ? 0.0 : (double)(-log2l((long double)inv));   // tab matches the ROUNDED inv
        }
        RB_CUDA(cudaMalloc(&F.d_log2i, sizeof(il)));
        RB_CUDA(cudaMemcpy(F.d_log2i, il, sizeof(il), cudaMemcpyHostToDevice));
    }
    for (int ap = 0; ap < 2; ++ap) {
        RB_CUDA(cudaMalloc(&F.d_pairpow[ap], sizeof(PairPow)));
        RB_CUDA(cudaMemcpy(F.d_pairpow[ap], &F.host.pair_pow[ap], sizeof(PairPow), cudaMemcpyHostToDevice));
    }
    return 0;
}

static int get_factor(long long n, double lam, FactorRef *out)
{
    int dev = 0;
    RB_CUDA(cudaGetDevice(&dev));
    const auto key = std::make_pair(n, lam);
    {
        std::lock_guard<std::mutex> lock(g_fmutex);
        auto &cache = g_fcache[dev & 15];
        auto it = cache.find(key);
        if (it != cache.end()) { it->second->last_use = ++g_fclock; *out = it->second; return 0; }
    }
    // build and upload outside the lock (first use costs a few synchronous copies); a racing thread may build the same
    // key, in which case the first one to publish wins and the other copy dies with its last reference
    FactorRef F = std::make_shared<FactorDev>();
    F->device = dev;
    build_factor(n, lam, F->host);
    RB_TRY(upload_factor(*F));
    std::lock_guard<std::mutex> lock(g_fmutex);
    auto &cache = g_fcache[dev & 15];
    auto it = cache.find(key);
    if (it != cache.end()) { it->second->last_use = ++g_fclock; *out = it->second; return 0; }
    while (cache.size() >= FACTOR_CACHE_MAX) {              // evict the least recently used entry nobody else holds
        auto victim = cache.end();
        for (auto e = cache.begin(); e != cache.end(); ++e)
            if (e->second.use_count() == 1 && (victim == cache.end() || e->second->last_use < victim->second->last_use)) victim = e;
        if (victim == cache.end()) break;                    // everything is in use: let the cache grow
        cache.erase(victim);
    }
    F->last_use = ++g_fclock;
    cache[key] = F;
    *out = F;
    return 0;
}

template <bool F32, int THREADS, int ITEMS, int CL>
static int launch_stream(PairParams R, long long pairs, cudaStream_t st)
{
    constexpr size_t sm = sizeof(double) * 2 * THREADS * ITEMS + sizeof(PairPow) + 16 * LOG2_V2_ENTRIES;
    auto kern = k_whittaker_stream<F32, THREADS, ITEMS, CL>;
    static bool attr_dev[64] = {false};
    static int resident_dev[64] = {0};
    int d = 0;
    cudaGetDevice(&d);
    bool &attr = attr_dev[d & 63];
    if (!attr) {
        RB_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm));
        RB_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributePreferredSharedMemoryCarveout, 100));
        attr = true;
    }
    cudaLaunchAttribute at{};
    at.id = cudaLaunchAttributeClusterDimension;
    at.val.clusterDim.x = CL; at.val.clusterDim.y = 1; at.val.clusterDim.z = 1;
    cudaLaunchConfig_t cfg{};
    cfg.blockDim = dim3(THREADS); cfg.dynamicSmemBytes = sm; cfg.stream = st; cfg.attrs = &at; cfg.numAttrs = 1;
    // persistent grid: as many clusters as are co-resident (1024 threads per SM)
    int &resident = resident_dev[d & 63];
    if (resident == 0) {
        cfg.gridDim = dim3((unsigned)(CL * sm_count()));
        int nc = 0;
        if (cudaOccupancyMaxActiveClusters(&nc, kern, &cfg) != cudaSuccess || nc <= 0) {
            (void)cudaGetLastError();
            nc = sm_count() * (1024 / THREADS) / CL;
        }
        resident = nc;
    }
    R.total_pairs = (int)pairs;
    R.w_y = R.write_baseline ? 0.0 : 1.0;
    R.w_b = R.write_baseline ? 0.5 : -0.5;
    const long long clusters = std::min<long long>(pairs, resident);
    cfg.gridDim = dim3((unsigned)(clusters * CL));
    RB_CUDA(cudaLaunchKernelEx(&cfg, kern, R));
    count_launch();
    return 0;
}

static long long gcd_ll(long long a, long long b) { while (b) { const long long t = a % b; a = b; b = t; } return a < 0 ? -a : a; }

int whittaker_rows(const void *d_x, int in_f32, int log_transform, const double *d_pilot, long long rows, long long n,
                   long long row_stride, double lam, int write_baseline, double *d_out, int *d_bad, cudaStream_t st)
{
    if (rows <= 0 || n <= 0) return ST_INVALID;
    const size_t esz = in_f32 ? 4 : 8;
    if (reinterpret_cast<uintptr_t>(d_x) % esz != 0) return ST_INVALID;      // every kernel loads whole elements
    WhitParams P{};
    P.x = d_x; P.pilot = d_pilot; P.out = d_out; P.bad = d_bad; P.n = n; P.row_stride = row_stride;
    P.rows = (int)rows; P.in_f32 = in_f32; P.log_transform = log_transform; P.write_baseline = write_baseline;
    if (n < 25) {
        const long long total = rows * n;
        const int blocks = (int)std::min<long long>((total + 255) / 256, 148 * 8);
        k_small_rows<<<blocks, 256, 0, st>>>(P);
        RB_LAUNCH_CHECK();
        return 0;
    }
    FactorRef F;                                       // keeps the host tables alive while this call reads them
    RB_TRY(get_factor(n, lam, &F));
    P.head_len = F->host.head_len;
    for (int p = 0; p < 2; ++p)
        for (int k = 0; k < 3; ++k) P.head[p][k] = F->d_head[p][k];
    memcpy(P.steady, F->host.steady, sizeof(P.steady));
    memcpy(P.tail, F->host.tail, sizeof(P.tail));
    P.log2tab = F->d_log2;
    if (!F->host.tiles_exact) return whittaker_exact(P, lam, st);
    P.tiles_per_row = (int)((n + WT_OUT - 1) / WT_OUT);
    // Interior tiles (region inside [head_len, n-4)) take the streaming kernel unless the penalty is too small for its
    // right-to-left re-derivation; the first and last tile(s) of each row take k_whittaker.  Launches over disjoint tile sets.
    const size_t sm_general = sizeof(double) * 2 * WT_THREADS_G * (WT_ITEMS_G + 1) + sizeof(double) * 6 * WT_THREADS_G;
    static bool attr_dev[64] = {false};
    int attr_d = 0;
    cudaGetDevice(&attr_d);
    bool &attr = attr_dev[attr_d & 63];
    if (!attr) {
        RB_CUDA(cudaFuncSetAttribute(k_whittaker<WT_THREADS_G, WT_ITEMS_G>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm_general));
        attr = true;
    }
    // classify tiles
    int first_steady = P.tiles_per_row, last_steady = -1;
    for (int t = 0; t < P.tiles_per_row; ++t) {
        const long long o0 = (long long)t * WT_OUT, o1 = std::min(n, o0 + WT_OUT);
        const long long r0 = std::max<long long>(0, o0 - WT_HALO), r1 = std::min(n, o1 + WT_HALO);
        const bool steady = F->host.stream_stable && (r0 >= P.head_len + 8) && (r1 <= n - 6) && (r1 - r0 == WT_REGION);      // (+8: room for the streaming kernel's alignment shift)
        if (steady) { first_steady = std::min(first_steady, t); last_steady = std::max(last_steady, t); }
    }
    // general tiles: [0, first_steady) and (last_steady, tiles); steady tiles are contiguous in between
    struct Span { int t0, t1; bool steady; };
    std::vector<Span> spans;
    if (last_steady >= first_steady) {
        if (first_steady > 0) spans.push_back({0, first_steady, false});
        spans.push_back({first_steady, last_steady + 1, true});
        if (last_steady + 1 < P.tiles_per_row) spans.push_back({last_steady + 1, P.tiles_per_row, false});
    } else {
        spans.push_back({0, P.tiles_per_row, false});
    }
    for (const Span &sp : spans) {
        WhitParams Q = P;
        Q.tile_offset = sp.t0;
        Q.span_tiles = sp.t1 - sp.t0;
        const long long blocks = rows * (long long)Q.span_tiles;
        if (blocks > 0x3fffffffLL) return ST_INVALID;
        // algorithmic bytes of this launch: read the input once, write the centered matrix once
        const double span_bins = (double)std::min<long long>(n, (long long)sp.t1 * WT_OUT) - (double)sp.t0 * WT_OUT;
        RB_PROF(sp.steady ? "k_whittaker_steady" : "k_whittaker_edge", st, (double)rows * span_bins * ((in_f32 ? 4.0 : 8.0) + 8.0));
        if (sp.steady) {
            // rows whose start has the same offset inside a 16-byte unit share a launch (the bulk copy needs an aligned source)
            const long long M = 16 / (long long)esz;
            const long long base_off = (long long)((reinterpret_cast<uintptr_t>(d_x) / esz) % (uintptr_t)M);
            const long long period = M / gcd_ll(row_stride % M, M);
            for (long long p = 0; p < period && p < rows; ++p) {
                PairParams R{};
                R.x = d_x; R.pilot = d_pilot; R.out = d_out; R.bad = d_bad; R.n = n; R.row_stride = row_stride;
                R.row0 = (int)p; R.row_step = (int)period; R.tile_offset = sp.t0; R.span_tiles = Q.span_tiles;
                R.shift = (int)((base_off + p * (row_stride % M)) % M);
                R.log_transform = log_transform; R.write_baseline = write_baseline;
                R.tab = F->host.pair_tab[R.shift & 1];
                R.pow_tab = F->d_pairpow[R.shift & 1];
                R.log2tab = F->d_log2i;
                const long long nrows = (rows - p + period - 1) / period;
                RB_TRY(in_f32 ? (launch_stream<true, WP_GEOM_THREADS, WP_GEOM_ITEMS, 2>(R, nrows * Q.span_tiles, st))
                              : (launch_stream<false, WP_GEOM_THREADS, WP_GEOM_ITEMS, 2>(R, nrows * Q.span_tiles, st)));
            }
        } else {
            k_whittaker<WT_THREADS_G, WT_ITEMS_G><<<(unsigned)blocks, WT_THREADS_G, sm_general, st>>>(Q);
            RB_LAUNCH_CHECK();
        }
    }
    // (kernels still in flight when an evicted entry dies are safe: cudaFree synchronises with the device first)
    return 0;
}

}  // namespace score
}  // namespace rb
