// Helpers shared by the nearest-neighbour scans (chamfer.cu, knn.cu): packed FP32x2 arithmetic, per-pair lengths of
// ragged batches, host-side validation of a cloud pair.  Holds no kernel, so any translation unit may include it.
#pragma once
#include "ptk_common.cuh"

namespace ptk {

typedef unsigned long long u64;

__device__ __forceinline__ u64 pack2(float lo, float hi) {
    u64 r;
    asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi));
    return r;
}
__device__ __forceinline__ void unpack2(u64 v, float &lo, float &hi) {
    asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(v));
}
__device__ __forceinline__ u64 fma2(u64 a, u64 b, u64 c) {
    u64 r;
    asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(r) : "l"(a), "l"(b), "l"(c));
    return r;
}
__device__ __forceinline__ u64 sub2(u64 a, u64 b) {
    u64 r;
    asm("sub.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b));
    return r;
}
__device__ __forceinline__ u64 mul2(u64 a, u64 b) {
    u64 r;
    asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b));
    return r;
}

// Ragged batches: the points of cloud b that exist, len[b] clamped to [0, P] (P when the caller passed no lengths).
// Row strides stay those of the padded (B, P, 3) tensor; only the counts of queries and targets become per pair, so
// padding points are never read into a result, a bound or the filter's certificate.
__device__ __forceinline__ int pair_len(const int64_t *__restrict__ len, int b, int P) {
    if (len == nullptr) return P;
    const long long v = len[b];
    return v < 0 ? 0 : (v > P ? P : (int)v);
}

// Fixed-order per-pair reductions (chamfer_finalize_kernel, the Chamfer normal term): a pair's queries are cut into
// fin_splits(l1, l2) slices of its OWN lengths, one CTA per slice, and the slice partials are added in slice order, so
// a pair's value depends neither on the batch nor on the padding it is computed in.  1 slice up to 16k points.
constexpr int FIN_SLICE = 16384;
__host__ __device__ inline int fin_splits(int64_t P1, int64_t P2) {
    const int64_t n = ceil_div(P1 > P2 ? P1 : P2, (int64_t)FIN_SLICE);
    return (int)(n < 1 ? 1 : (n > 64 ? 64 : n));
}

// cham[b] from the two sums: mean = sum_x / max(lx, 1) + sum_y / max(ly, 1), sum = sum_x + sum_y
__device__ __forceinline__ float chamfer_reduce(float sx, float sy, int L1, int L2, int mean) {
    return mean ? sx / (float)max(L1, 1) + sy / (float)max(L2, 1) : sx + sy;
}

// host-side validation of a cloud pair shared by the Chamfer and K-NN entry points
static inline int check_clouds(const void *x, const void *y, int64_t B, int64_t P1, int64_t P2) {
    PTK_REQUIRE(x && y, PTK_ERR_SHAPE, "chamfer: null cloud pointer");
    PTK_REQUIRE(B > 0 && P1 > 0 && P2 > 0, PTK_ERR_SHAPE,
                "chamfer: empty input (B=%lld, P1=%lld, P2=%lld); point clouds must be non-empty",
                (long long)B, (long long)P1, (long long)P2);
    PTK_REQUIRE(P1 < (1LL << 31) / 3 && P2 < (1LL << 31) / 3, PTK_ERR_SHAPE,
                "chamfer: cloud too large for 32-bit indexing");
    return PTK_OK;
}

}  // namespace ptk
