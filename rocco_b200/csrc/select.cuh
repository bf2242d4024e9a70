// Radix SELECT inside a thread block (shared by the trend's slot / bin selections and the pilot offsets).
#pragma once
#include "common.cuh"

namespace rb {
namespace score {

// Only one or two order statistics of a slot are ever wanted, so the slot is not sorted: an MSB-first radix SELECT over
// the keys in shared memory (11 bits per pass, starting at the highest bit in which the keys differ) finds the key of a
// given rank in two or three passes of `cnt / THREADS` elements per thread, where the bitonic sort needs ~log2(cnt)^2 / 2.
constexpr int SEL_BITS = 11, SEL_BINS = 1 << SEL_BITS;

struct SelScratch { int hist[SEL_BINS]; unsigned long long res[4]; int ires[4]; };
__device__ __forceinline__ SelScratch &plan_scratch(void *raw) { return *reinterpret_cast<SelScratch *>(raw); }

// Key of 0-based `rank` among the keys[i], i < cnt, that pass the filter (fkeys == nullptr, or fkeys[i] == fval).  All
// THREADS threads call it; the result is uniform.  *below = number of filtered keys smaller than the result, *equal =
// number equal to it.  The filtered set must hold more than `rank` keys.
// RENARROW: after each pass, the next one starts at the highest bit in which the remaining candidates differ, and a
// bucket of equal keys ends the search -- one extra scan per pass, but a column of tied values (mostly zeros in count
// data) takes two scans instead of falling through every digit.
template <int THREADS, bool RENARROW = false>
__device__ unsigned long long block_select(const unsigned long long *keys, int cnt, int rank, const unsigned long long *fkeys,
                                           unsigned long long fval, SelScratch &S, int *below, int *equal)
{
    const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    // highest differing bit of the filtered keys
    unsigned long long kmin = ~0ULL, kmax = 0ULL;
    for (int i = tid; i < cnt; i += THREADS)
        if (!fkeys || fkeys[i] == fval) { const unsigned long long k = keys[i]; kmin = min(kmin, k); kmax = max(kmax, k); }
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) {
        kmin = min(kmin, __shfl_xor_sync(0xffffffffu, kmin, d));
        kmax = max(kmax, __shfl_xor_sync(0xffffffffu, kmax, d));
    }
    __syncthreads();                                       // S may still be read by a previous call
    if (tid == 0) { S.res[0] = ~0ULL; S.res[1] = 0ULL; }
    __syncthreads();
    if (lane == 0) { atomicMin(&S.res[0], kmin); atomicMax(&S.res[1], kmax); }
    __syncthreads();
    kmin = S.res[0]; kmax = S.res[1];
    int top = 64 - __clzll((long long)(kmin ^ kmax));      // number of low bits that can differ (0: all keys equal)
    unsigned long long prefix = (top >= 64) ? 0ULL : (kmin >> top) << top, mask = (top >= 64) ? 0ULL : ~((1ULL << top) - 1ULL);
    int r = rank, nbelow = 0, nequal = 0;
    bool found = false;
    unsigned long long result = kmin;
    if (top == 0) {                                        // every filtered key is the same value
        int c = 0;
        for (int i = tid; i < cnt; i += THREADS) c += (!fkeys || fkeys[i] == fval);
#pragma unroll
        for (int d = 16; d > 0; d >>= 1) c += __shfl_xor_sync(0xffffffffu, c, d);
        __syncthreads();
        if (tid == 0) S.ires[0] = 0;
        __syncthreads();
        if (lane == 0) atomicAdd(&S.ires[0], c);
        __syncthreads();
        nequal = S.ires[0];
        found = true;
    }
    while (!found) {
        const int width = min(SEL_BITS, top), shift = top - width;
        for (int k = tid; k < SEL_BINS; k += THREADS) S.hist[k] = 0;
        __syncthreads();
        for (int i = tid; i < cnt; i += THREADS) {
            const unsigned long long k = keys[i];
            if ((!fkeys || fkeys[i] == fval) && (k & mask) == prefix) atomicAdd(&S.hist[(int)((k >> shift) & (unsigned long long)((1 << width) - 1))], 1);
        }
        __syncthreads();
        if (wid == 0) {                                    // digit whose cumulative count passes r: 64 bins per lane
            int sum = 0;
            for (int k = 0; k < SEL_BINS / 32; ++k) sum += S.hist[lane * (SEL_BINS / 32) + k];
            int inc = sum;
#pragma unroll
            for (int d = 1; d < 32; d <<= 1) { const int o = __shfl_up_sync(0xffffffffu, inc, d); if (lane >= d) inc += o; }
            const int exc = inc - sum;
            if (exc <= r && r < inc) {
                int acc = exc, k = 0;
                for (; k < SEL_BINS / 32; ++k) { const int h = S.hist[lane * (SEL_BINS / 32) + k]; if (r < acc + h) break; acc += h; }
                S.ires[0] = lane * (SEL_BINS / 32) + k; S.ires[1] = acc; S.ires[2] = S.hist[lane * (SEL_BINS / 32) + k];
            }
        }
        __syncthreads();
        const int digit = S.ires[0], before = S.ires[1], inside = S.ires[2];
        nbelow += before; r -= before;
        prefix |= (unsigned long long)digit << shift;
        mask |= (unsigned long long)((1 << width) - 1) << shift;
        top = shift;
        if (top == 0) { result = prefix; nequal = inside; found = true; }
        else if (inside == 1) {                            // a single candidate left: fetch it
            for (int i = tid; i < cnt; i += THREADS) {
                const unsigned long long k = keys[i];
                if ((!fkeys || fkeys[i] == fval) && (k & mask) == prefix) S.res[2] = k;
            }
            __syncthreads();
            result = S.res[2]; nequal = 1; found = true;
        } else if (RENARROW) {
            unsigned long long cmin = ~0ULL, cmax = 0ULL;
            for (int i = tid; i < cnt; i += THREADS) {
                const unsigned long long k = keys[i];
                if ((!fkeys || fkeys[i] == fval) && (k & mask) == prefix) { cmin = min(cmin, k); cmax = max(cmax, k); }
            }
#pragma unroll
            for (int d = 16; d > 0; d >>= 1) {
                cmin = min(cmin, __shfl_xor_sync(0xffffffffu, cmin, d));
                cmax = max(cmax, __shfl_xor_sync(0xffffffffu, cmax, d));
            }
            if (tid == 0) { S.res[0] = ~0ULL; S.res[1] = 0ULL; }          // S.res[0..1] were last read before the histogram
            __syncthreads();
            if (lane == 0) { atomicMin(&S.res[0], cmin); atomicMax(&S.res[1], cmax); }
            __syncthreads();
            cmin = S.res[0]; cmax = S.res[1];
            const int t2 = 64 - __clzll((long long)(cmin ^ cmax));       // < top: the candidates share the prefix
            if (t2 == 0) { result = cmin; nequal = inside; found = true; }
            else { top = t2; prefix = (cmin >> top) << top; mask = ~((1ULL << top) - 1ULL); }
        }
        __syncthreads();
    }
    if (below) *below = nbelow;
    if (equal) *equal = nequal;
    return result;
}

}  // namespace score
}  // namespace rb
