// Internal interfaces between the scoring translation units.
#pragma once
#include "common.cuh"

namespace rb {
namespace score {

// Cross-fit Whittaker baseline over `rows` rows of length n (row-major, `row_stride` elements apart).
// log_transform: y = log2(max(x,0)+1) - pilot[row];  write_baseline: out = baseline, else out = y - baseline.
int whittaker_rows(const void *d_x, int in_f32, int log_transform, const double *d_pilot, long long rows, long long n,
                   long long row_stride, double lam, int write_baseline, double *d_out, int *d_bad, cudaStream_t st);
// Rows solved by the exact sequential path (penalties beyond the tile kernels' range, whittaker.cu) since load.
long long whittaker_exact_rows();

// Pilot offsets: per-row median of log2(max(x,0)+1) -- exact for n <= 4096, else the median of a
// 4096-point strided sample (the offset cancels in  y - baseline(y)  up to the solver's noise).
// exact != 0: np.median for any n (one radix sort per row).
int pilot_offsets(const void *d_x, int in_f32, long long rows, long long n, long long row_stride, double *d_pilot,
                  cudaStream_t st, int exact = 0);

// Centered matrix -> per-locus WLS outputs (wls_backend.c:744-947).  d_acc2 != nullptr: stop at the column sums of these
// rows instead, d_acc2[2][n] = {sum y/post, sum 1/post} (what scores and mean need), for finalize_acc after a cross-rank sum.
int centered_wls(const double *d_centered, long long m, long long n, const rocco_b200_score_params &prm,
                 rocco_b200_score_outputs *out, cudaStream_t st, double *d_acc2 = nullptr);

// Per-bin outputs from column sums over m_total samples (wls_backend.c:915-937): d_acc [4][n], or [2][n] without has_rq (the
// raw / prior variance outputs must then be NULL).  Sets *d_bad on a non-finite result.
int finalize_acc(const double *d_acc, long long n, bool has_rq, long long m_total, const rocco_b200_score_params &prm,
                 rocco_b200_score_outputs *out, int *d_bad, cudaStream_t st);

// a / b from a correctly rounded reciprocal rb = RN(1/b): Markstein's final step (q = RN(a*rb), r = a - q*b exactly by
// FMA, RN(q + r*rb)) gives the correctly rounded quotient for operands in the normal range without the generic
// division's special-case slow path (~3 issue slots instead of ~30).
__device__ __forceinline__ double div_rcp(double a, double b, double rb)
{
    const double q = __dmul_rn(a, rb);
    const double r = __fma_rn(-q, b, a);
    return __fma_rn(r, rb, q);
}

// 1 / d for d in the normal range: hardware seed (MUFU.RCP64H, ~20 bits) and two Newton steps (~1 ulp), without the
// generic division's special-case slow path.
__device__ __forceinline__ double rcp_nr(double d)
{
    double r;
    asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(r) : "d"(d));
    double e = __fma_rn(-d, r, 1.0);
    r = __fma_rn(r, e, r);
    e = __fma_rn(-d, r, 1.0);
    return __fma_rn(r, e, r);
}

// AR(1) innovation variance of one window from its three sums (wls_backend.c:665-712).  The algebra is the reference's;
// the operations are fused (FMA) and regrouped:  g1 = sl - mu (sum_head + sum_tail) + pairs mu^2,
// denom = g0 (1 + lambda_eff) + 1e-4 (g0 + 1) = g0 c1 + 1e-4 with c1 = 1 + lambda_eff + 1e-4 (always > eps = 1e-12 (g0 + 1), so
// the reference's guard never fires), beta = g1 / denom by reciprocal.  Differences from the reference's own rounding
// are ~1e-16 relative per operation, far below the ~1e-12 drift of its whole-row sliding sums.
// rwd = 1/wd, c1 as above.
__device__ __forceinline__ double ar1_window_variance(double s1, double s2, double sl, double first, double last, double wd,
                                                      double rwd, double pairs, double c1)
{
    const double mu = s1 * rwd;
    const double g0 = dmax(__fma_rn(-(wd * mu), mu, s2), 0.0);
    const double g1 = __fma_rn(pairs * mu, mu, __fma_rn(-mu, (s1 - last) + (s1 - first), sl));
    const double den = __fma_rn(g0, c1, 1.0e-4);
    double beta = g1 * rcp_nr(den);
    beta = dmin(dmax(beta, 0.0), 0.99);
    return (g0 * rwd) * __fma_rn(-beta, beta, 1.0);
}

int resolve_spatial_window(long long n, int requested);
int resolve_baseline_window(long long n, int target);
double whittaker_lambda(int block);

}  // namespace score
}  // namespace rb
