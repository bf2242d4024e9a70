// Trend-knot interfaces shared by trend.cu (histogram multi-select) and wls.cu (sort-based path, combine).
#pragma once
#include "common.cuh"

namespace rb {
namespace score {

constexpr int MAX_KNOTS = 64;

struct Knots { double x[MAX_KNOTS]; double y[MAX_KNOTS]; int nk; int constant; double cval; };

// bin medians -> PAVA -> de-duplicated knots (wls_backend.c:507-560, 262-338); single thread
__device__ void knots_from_bins(const double *bx, const double *by, const double *bw, int used, Knots *out);

// Histogram multi-select for all m rows; rows it cannot handle (a bucket over capacity) get row_fallback = 1.
// fused_window > 0: d_V is an OUTPUT -- the rolling AR(1) variance (window `fused_window`, already resolved) is
// computed in the same pass as the first histogram, which also writes a 32-bit key per pair (4 B per sample-bin of
// scratch) that the slot collection reads instead of C and V; fused_window == 0: d_V is an input.
int trend_knots_select(const double *d_C, double *d_V, long long m, long long n, long long row_stride, Knots *d_knots,
                       int *d_row_fallback, int fused_window, cudaStream_t st);
int trend_fused_max_window();

}  // namespace score
}  // namespace rb
