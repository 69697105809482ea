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
//
// Every _det backward runs the same three phases on the same workspace (the helpers below):
//   1. M_b: atomicMax of the largest finite |term| into mbits[b] (det_block_max), each row's accumulator and output
//      zeroed (det_zero_row);
//   2. every term added to its row (det_add);
//   3. det_convert_kernel: each row's gradient from its sum.
// Phases 2 and 3 read e_b from the same DetBound, so they cannot disagree on n.
#pragma once
#include "nn_common.cuh"

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

__device__ __forceinline__ float det_abs_finite(float t) { return isfinite(t) ? fabsf(t) : 0.0f; }

// n_b, the bound on the terms one row of batch element b receives (+ 1): max(l_a, l_b) + add, where l_a / l_b are the
// element's lengths in the ragged sense of pair_len (an absent length is (NULL, 0): pair_len gives 0).  A constant
// bound is add alone.
struct DetBound {
    const int64_t *len_a, *len_b;
    int P_a, P_b;
    long long add;
    __device__ __forceinline__ long long n(int b) const {
        return (long long)max(pair_len(len_a, b, P_a), pair_len(len_b, b, P_b)) + add;
    }
};
inline DetBound det_bound_len(const int64_t *len_a, int64_t P_a, const int64_t *len_b = nullptr, int64_t P_b = 0) {
    return DetBound{len_a, len_b, (int)P_a, (int)P_b, 1};
}
inline DetBound det_bound_const(long long n) { return DetBound{nullptr, nullptr, 0, 0, n}; }

// 2^e_b for phase 2
__device__ __forceinline__ double det_scale(const unsigned int *mbits, const DetBound &nb, int b) {
    return ldexp(1.0, det_exponent(mbits[b], nb.n(b)));
}

// phase 1: row r (3 components) of an accumulator and of its output
__device__ __forceinline__ void det_zero_row(unsigned long long *acc, float *out, size_t r) {
    acc[r * 3 + 0] = acc[r * 3 + 1] = acc[r * 3 + 2] = 0ull;
    out[r * 3 + 0] = out[r * 3 + 1] = out[r * 3 + 2] = 0.0f;
}

// phase 2: one term into one component: Q(t) into the accumulator (global or shared) when t is finite, otherwise t
// into the output.  A term that goes in negated is passed as -t: round-half-even is symmetric, so Q(-t) = -Q(t).
__device__ __forceinline__ void det_add(unsigned long long *acc, float *out, float t, double scale) {
    if (isfinite(t))
        atomicAdd(acc, det_quantise(t, scale));
    else
        atomicAdd(out, t);
}

// phase 3, grid = (ceil(max(rows_a, rows_b) / THREADS), B): row i of out_a and of out_b (either may be NULL) =
// fp32(acc) * 2^-e_b, unless the output already holds a non-finite sum
template <int THREADS>
__global__ void __launch_bounds__(THREADS)
det_convert_kernel(DetBound nb, const unsigned int *__restrict__ mbits, const unsigned long long *__restrict__ acc_a,
                   float *__restrict__ out_a, int rows_a, const unsigned long long *__restrict__ acc_b,
                   float *__restrict__ out_b, int rows_b) {
    pdl_wait();
    const int b = blockIdx.y;
    const int i = blockIdx.x * THREADS + threadIdx.x;
    const int e = det_exponent(mbits[b], nb.n(b));
    if (out_a && i < rows_a) {
        const size_t r = ((size_t)b * rows_a + i) * 3;
        for (int d = 0; d < 3; ++d)
            if (isfinite(out_a[r + d])) out_a[r + d] = ldexpf(__ll2float_rn((long long)acc_a[r + d]), -e);
    }
    if (out_b && i < rows_b) {
        const size_t r = ((size_t)b * rows_b + i) * 3;
        for (int d = 0; d < 3; ++d)
            if (isfinite(out_b[r + d])) out_b[r + d] = ldexpf(__ll2float_rn((long long)acc_b[r + d]), -e);
    }
}

// ---- host side.  Workspace: [M_b bits, 4 B per element, padded to 256 B][acc_a: 24 B per row a], then, when there
// are rows b, [padding to 256 B][acc_b: 24 B per row b].  rows_a / rows_b: the rows of one batch element.
inline size_t det_align(size_t b) { return (b + 255) & ~(size_t)255; }

inline size_t det_workspace_bytes(int64_t B, int64_t rows_a, int64_t rows_b = 0) {
    const size_t a = 24 * (size_t)B * (size_t)rows_a;
    return det_align(4 * (size_t)B) + (rows_b > 0 ? det_align(a) + 24 * (size_t)B * (size_t)rows_b : a);
}

// the workspace check of every _det entry point
inline int det_check_workspace(const void *ws, size_t bytes, size_t need, const char *what) {
    PTK_REQUIRE(ws && bytes >= need, PTK_ERR_WORKSPACE, "%s: workspace too small (%zu < %zu)", what, bytes, need);
    PTK_REQUIRE((reinterpret_cast<uintptr_t>(ws) & 15) == 0, PTK_ERR_ALIGN, "%s: workspace must be 16-byte aligned",
                what);
    return PTK_OK;
}

struct DetWs {
    unsigned int *mbits;
    unsigned long long *acc_a, *acc_b;
};

// the sections of a det_workspace_bytes(B, rows_a, ...) workspace, with M_b zeroed on st (the one memset)
inline cudaError_t det_begin(void *ws, int64_t B, int64_t rows_a, cudaStream_t st, DetWs &w) {
    char *p = reinterpret_cast<char *>(ws);
    const size_t m = det_align(4 * (size_t)B);
    w.mbits = reinterpret_cast<unsigned int *>(p);
    w.acc_a = reinterpret_cast<unsigned long long *>(p + m);
    w.acc_b = reinterpret_cast<unsigned long long *>(p + m + det_align(24 * (size_t)B * (size_t)rows_a));
    return cudaMemsetAsync(w.mbits, 0, sizeof(unsigned int) * (size_t)B, st);
}

// phase 3 launch (rows of out_b: 0 when there is one output)
template <int THREADS>
inline cudaError_t det_launch_convert(const DetWs &w, const DetBound &nb, int64_t B, float *out_a, int64_t rows_a,
                                      float *out_b, int64_t rows_b, cudaStream_t st) {
    const int64_t rows = rows_a > rows_b ? rows_a : rows_b;
    return launch_pdl(det_convert_kernel<THREADS>, dim3((unsigned)ceil_div(rows, THREADS), (unsigned)B), dim3(THREADS), 0,
                      st, nb, (const unsigned int *)w.mbits, (const unsigned long long *)w.acc_a, out_a, (int)rows_a,
                      (const unsigned long long *)w.acc_b, out_b, (int)rows_b);
}

}  // namespace ptk
