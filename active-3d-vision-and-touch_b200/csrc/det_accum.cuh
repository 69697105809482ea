// Deterministic backward: exact fixed-point accumulation of fp32 gradient terms (DESIGN.md K1 / K3, include/ptk.h).
//
// A scatter-add whose rows receive terms in scheduling order gives different fp32 bits from run to run.  The _det
// backward kernels instead quantise every finite term t of a batch element b to
//     Q(t) = round_half_even(t * 2^e_b)  (an int64; the product is exact in double)
//     e_b  = 62 - ceil(log2 M_b) - ceil(log2 n)
// where M_b is the largest finite |term| of b and n bounds the number of terms one row can receive (+ 1).  Every
// |Q(t)| <= 2^(62 - ceil(log2 n)), so a row's sum stays below 2^62: 64-bit integer atomics add it exactly, in any
// order.  The row's gradient is fp32(sum) * 2^-e_b: one round-to-nearest-even rounding of the exact quantised sum.
// Non-finite terms bypass the integer sum and are added (fp32 atomics, order-free: only non-finite values meet there)
// to the row's output, which the conversion leaves alone when it is not finite.
#pragma once
#include "ptk_common.cuh"

namespace ptk {

// smallest c with 2^c >= v, for a finite v > 0 given by its bit pattern
__device__ __forceinline__ int det_ceil_log2_bits(unsigned int bits) {
    const int E = (int)(bits >> 23);
    const unsigned int f = bits & 0x7fffffu;
    if (E == 0) return -149 + (32 - __clz((int)(f - 1u)));  // subnormal: v = f * 2^-149
    return f == 0u ? E - 127 : E - 126;
}

// smallest c with 2^c >= n (n >= 1)
__host__ __device__ inline int det_ceil_log2_int(long long n) {
    int c = 0;
    while ((1LL << c) < n) ++c;
    return c;
}

// e_b from the bit pattern of M_b (0: every finite term is zero, e_b = 0) and the term bound n
__device__ __forceinline__ int det_exponent(unsigned int mbits, long long n) {
    return mbits == 0u ? 0 : 62 - det_ceil_log2_bits(mbits) - det_ceil_log2_int(n);
}

// Q(t) for a finite t; scale = 2^e_b (exact: |e_b| stays far inside the double range)
__device__ __forceinline__ unsigned long long det_quantise(float t, double scale) {
    return (unsigned long long)__double2ll_rn((double)t * scale);
}

// largest finite |t| of the block -> atomicMax on the bit pattern (non-negative floats order like unsigned ints)
template <int THREADS>
__device__ __forceinline__ void det_block_max(float m, unsigned int *mbits) {
    __shared__ float red[THREADS / 32];
    m = warp_max(m);
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = m;
    __syncthreads();
    if (threadIdx.x == 0) {
        float v = red[0];
        for (int w = 1; w < THREADS / 32; ++w) v = fmaxf(v, red[w]);
        if (v > 0.0f) atomicMax(mbits, __float_as_uint(v));
    }
}

// workspace sections are aligned to 256 bytes
inline size_t det_align(size_t b) { return (b + 255) & ~(size_t)255; }

__device__ __forceinline__ float det_abs_finite(float t) { return isfinite(t) ? fabsf(t) : 0.0f; }

// the row's gradient: its output holds the sum of its non-finite terms (0 when there are none)
__device__ __forceinline__ void det_convert(float *out, const unsigned long long *acc, int e) {
    if (isfinite(*out)) *out = ldexpf(__ll2float_rn((long long)*acc), -e);
}

}  // namespace ptk
