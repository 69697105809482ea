// Helpers shared by the nearest-neighbour scans (chamfer.cu, knn.cu): the defining distance arithmetic in scalar and
// packed FP32x2 form, the shared-memory tile stager, per-pair lengths of ragged batches, host-side validation of a
// cloud pair.  Holds no kernel, so any translation unit may include it.
#pragma once
#include "ptk_common.cuh"

namespace ptk {

typedef unsigned long long u64;

constexpr int CH_TT = 2048;   // targets per shared-memory tile of the exact scans (3 * 2048 * 4 B = 24 KB)

__device__ __forceinline__ float min3f(float a, float b, float c) {
    float r;
    asm("min.f32 %0, %1, %2, %3;" : "=f"(r) : "f"(a), "f"(b), "f"(c));
    return r;
}

// The one and only definition of the distance arithmetic (inner loop AND index recovery).
__device__ __forceinline__ float sqdist(float qx, float qy, float qz, float tx, float ty, float tz) {
    float dx = __fsub_rn(qx, tx);
    float dy = __fsub_rn(qy, ty);
    float dz = __fsub_rn(qz, tz);
    float d = __fmul_rn(dx, dx);
    d = __fmaf_rn(dy, dy, d);
    d = __fmaf_rn(dz, dz, d);
    return d;
}

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

// sqdist() of one query against four consecutive targets on packed FP32x2, two targets per instruction.  qx/qy/qz hold
// the query coordinate in both halves (pack2(q, q)); tx/ty/tz are the targets' coordinates as two packed pairs each.
// Contract: d0..d3 are sqdist()'s bits for the four targets -- every lane runs sqdist()'s sub, mul, fma, fma sequence
// with the same rounding -- so an index recovered with sqdist() finds the minimum the scan saw.
__device__ __forceinline__ void sqdist4(u64 qx, u64 qy, u64 qz, ulonglong2 tx, ulonglong2 ty, ulonglong2 tz, float &d0,
                                        float &d1, float &d2, float &d3) {
    const u64 dxa = sub2(qx, tx.x), dxb = sub2(qx, tx.y);
    const u64 dya = sub2(qy, ty.x), dyb = sub2(qy, ty.y);
    const u64 dza = sub2(qz, tz.x), dzb = sub2(qz, tz.y);
    u64 da = mul2(dxa, dxa), db = mul2(dxb, dxb);
    da = fma2(dya, dya, da);
    db = fma2(dyb, dyb, db);
    da = fma2(dza, dza, da);
    db = fma2(dzb, dzb, db);
    unpack2(da, d0, d1);
    unpack2(db, d2, d3);
}

// One tile of n targets, global (n,3) packed floats -> shared SoA sx[], sy[], sz[], padded with +inf to a whole number
// of CHUNK-target chunks (a padded target never wins '<' and never enters a K-NN list: its distance is +inf or NaN).
// Returns the tile's chunk count.  Eight loads in flight per thread: when only a few CTAs are resident (the rescue
// pass in list mode) this staging is latency-bound unless the loads are batched (ncu: 255 us rescue pass, long-
// scoreboard stalls).  The caller brackets it with __syncthreads().
template <int THREADS, int CHUNK>
__device__ __forceinline__ int stage_tile_soa(const float *__restrict__ src, int n, float *sx, float *sy, float *sz) {
    const int tid = threadIdx.x;
    const float INF = __int_as_float(0x7f800000);
    const int npad = ((n + CHUNK - 1) / CHUNK) * CHUNK;
    for (int e0 = 0; e0 < npad * 3; e0 += THREADS * 8) {
        float v[8];
#pragma unroll
        for (int u = 0; u < 8; ++u) {
            const int e = e0 + u * THREADS + tid;
            v[u] = e < n * 3 ? src[e] : INF;
        }
#pragma unroll
        for (int u = 0; u < 8; ++u) {
            const int e = e0 + u * THREADS + tid;
            if (e < npad * 3) {
                const int p = e / 3;
                const int c = e - p * 3;
                float *dst = c == 0 ? sx : (c == 1 ? sy : sz);
                dst[p] = v[u];
            }
        }
    }
    return npad / CHUNK;
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
