// Exact K nearest neighbours (1 <= K <= PTK_KNN_MAX_K) for sm_100a: pytorch3d.ops.knn_points for K > 1.
// Contract in include/ptk.h (ptk_knn_fwd_lengths): the K smallest (d, j) in lexicographic order, d = sqdist(); column 0
// is ptk_knn1_fwd_lengths' result bit for bit.  Design in DESIGN.md K1c: a brute-force scan with the 6-op arithmetic on
// packed FP32x2 (no filter: exact by construction), sorted lists in registers, chunks that can improve a list queued
// per query and drained per warp, target-range splits merged lexicographically for small batches.
#include <algorithm>

#include "nn_common.cuh"
#include "det_accum.cuh"

namespace ptk {

constexpr int KNN_THREADS = 128;
constexpr int KNN_CHUNK = 8;        // targets per chunk minimum
constexpr int KNN_QUEUE = 16;       // queued chunks per query before the warp drains
constexpr int KNN_MAX_SPLIT = 8;    // target-range splits merged by knn_merge_kernel
constexpr int KNN_MIN_SPLIT_LEN = 1024;
constexpr int64_t KNN_FILL_CTAS = 1024;  // split the targets while the query blocks alone give fewer CTAs

// queries per thread and resident CTAs per SM of each K bucket (the list costs 2 * KB registers per query)
__host__ __device__ constexpr int knn_bucket(int K) { return K <= 2 ? 2 : K <= 4 ? 4 : K <= 8 ? 8 : K <= 16 ? 16 : K <= 32 ? 32 : 64; }
__host__ __device__ constexpr int knn_rows(int KB) { return KB <= 16 ? 2 : 1; }
__host__ __device__ constexpr int knn_minb(int KB) { return KB <= 16 ? 4 : KB == 32 ? 3 : 2; }

// (d, j) into the ascending list (ld, lj), after every slot whose distance is <= d; the last slot drops out.
// The caller has checked d < ld[KB - 1].
template <int KB>
__device__ __forceinline__ void knn_insert(float (&ld)[KB], int (&lj)[KB], float d, int j) {
#pragma unroll
    for (int k = KB - 1; k > 0; --k) {
        const bool up = ld[k - 1] > d;  // slot k - 1 moves to k
        const bool here = ld[k] > d;    // first slot above d takes it
        ld[k] = up ? ld[k - 1] : (here ? d : ld[k]);
        lj[k] = up ? lj[k - 1] : (here ? j : lj[k]);
    }
    const bool here = ld[0] > d;
    ld[0] = here ? d : ld[0];
    lj[0] = here ? j : lj[0];
}

// grid = (ceil(P1 / (KNN_THREADS * R)), n_split, B).  n_split == 1: writes dist / idx (B,P1,K) with the zero fill;
// otherwise the split's sorted list of every valid query to part[b][split][i][K] (as (dist bits, idx)).
template <int KB, int R, int MINB>
__global__ void __launch_bounds__(KNN_THREADS, MINB)
knn_scan_kernel(const float *__restrict__ p1, const float *__restrict__ p2, const int64_t *__restrict__ len1,
                const int64_t *__restrict__ len2, int P1, int P2, int K, int split_len, int n_split,
                float *__restrict__ dist, int32_t *__restrict__ idx, uint2 *__restrict__ part) {
    pdl_wait();
    const int b = blockIdx.z;
    const int L1 = pair_len(len1, b, P1), L2 = pair_len(len2, b, P2);
    const int tid = threadIdx.x;
    const int q0 = blockIdx.x * (KNN_THREADS * R);
    const int t_begin = blockIdx.y * split_len;
    if (q0 >= L1 || t_begin >= L2) {
        // nothing to scan: the zero fill of padded queries and of pairs with an empty target cloud (unsplit launch;
        // with splits the merge kernel fills, and reads no list of a split past l2)
        if (n_split == 1)
            for (int r = 0; r < R; ++r) {
                const int qi = q0 + r * KNN_THREADS + tid;
                if (qi >= P1) break;
                for (int k = 0; k < K; ++k) {
                    dist[((size_t)b * P1 + qi) * K + k] = 0.0f;
                    idx[((size_t)b * P1 + qi) * K + k] = 0;
                }
            }
        return;
    }
    const int t_end = min(L2, t_begin + split_len);
    const float INF = __int_as_float(0x7f800000);
    const float *__restrict__ Q = p1 + (size_t)b * P1 * 3;
    const float *__restrict__ T = p2 + (size_t)b * P2 * 3;

    __shared__ __align__(16) float sx[CH_TT];
    __shared__ __align__(16) float sy[CH_TT];
    __shared__ __align__(16) float sz[CH_TT];
    __shared__ int queue[KNN_QUEUE][R][KNN_THREADS];  // tile-local chunk ids; [slot][row][thread]: conflict-free

    u64 qx[R], qy[R], qz[R];
    float ld[R][KB];
    int lj[R][KB], cnt[R];
#pragma unroll
    for (int r = 0; r < R; ++r) {
        const int qi = min(q0 + r * KNN_THREADS + tid, L1 - 1);
        const float a = Q[(size_t)qi * 3 + 0], bq = Q[(size_t)qi * 3 + 1], c = Q[(size_t)qi * 3 + 2];
        qx[r] = pack2(a, a);
        qy[r] = pack2(bq, bq);
        qz[r] = pack2(c, c);
#pragma unroll
        for (int k = 0; k < KB; ++k) {
            ld[r][k] = k < KB - K ? -INF : INF;
            lj[r][k] = 0;
        }
        cnt[r] = 0;
    }

    // re-evaluate every queued chunk of this tile in ascending j and insert what beats the current threshold
    auto drain = [&](int tile) {
#pragma unroll
        for (int r = 0; r < R; ++r) {
            float a, bq, c, dummy;
            unpack2(qx[r], a, dummy);
            unpack2(qy[r], bq, dummy);
            unpack2(qz[r], c, dummy);
            for (int e = 0; e < cnt[r]; ++e) {
                const int j0 = queue[e][r][tid] * KNN_CHUNK;
#pragma unroll 1
                for (int u = 0; u < KNN_CHUNK; ++u) {
                    const float d = sqdist(a, bq, c, sx[j0 + u], sy[j0 + u], sz[j0 + u]);
                    if (d < ld[r][KB - 1]) knn_insert<KB>(ld[r], lj[r], d, tile + j0 + u);
                }
            }
            cnt[r] = 0;
        }
    };

    for (int tile = t_begin; tile < t_end; tile += CH_TT) {
        const int n = min(CH_TT, t_end - tile);
        __syncthreads();
        const int nchunks = stage_tile_soa<KNN_THREADS, KNN_CHUNK>(T + (size_t)tile * 3, n, sx, sy, sz);
        __syncthreads();
        for (int ch = 0; ch < nchunks; ++ch) {
            float m[R];
#pragma unroll
            for (int r = 0; r < R; ++r) m[r] = INF;
#pragma unroll
            for (int g = 0; g < KNN_CHUNK / 4; ++g) {
                const ulonglong2 tx = *reinterpret_cast<const ulonglong2 *>(&sx[ch * KNN_CHUNK + g * 4]);
                const ulonglong2 ty = *reinterpret_cast<const ulonglong2 *>(&sy[ch * KNN_CHUNK + g * 4]);
                const ulonglong2 tz = *reinterpret_cast<const ulonglong2 *>(&sz[ch * KNN_CHUNK + g * 4]);
#pragma unroll
                for (int r = 0; r < R; ++r) {
                    float d0, d1, d2, d3;
                    sqdist4(qx[r], qy[r], qz[r], tx, ty, tz, d0, d1, d2, d3);
                    m[r] = min3f(m[r], d0, d1);
                    m[r] = min3f(m[r], d2, d3);
                }
            }
            int full = 0;
#pragma unroll
            for (int r = 0; r < R; ++r) {
                queue[cnt[r]][r][tid] = ch;  // overwritten unless the chunk can improve the list
                cnt[r] += m[r] < ld[r][KB - 1] ? 1 : 0;
                full |= cnt[r] == KNN_QUEUE;
            }
            if (__any_sync(0xffffffffu, full)) drain(tile);
        }
        drain(tile);  // before the tile is overwritten
    }

#pragma unroll
    for (int r = 0; r < R; ++r) {
        const int qi = q0 + r * KNN_THREADS + tid;
        if (qi >= L1) {
            if (n_split == 1 && qi < P1)
                for (int k = 0; k < K; ++k) {
                    dist[((size_t)b * P1 + qi) * K + k] = 0.0f;
                    idx[((size_t)b * P1 + qi) * K + k] = 0;
                }
            continue;
        }
        if (n_split == 1) {
            float *od = dist + ((size_t)b * P1 + qi) * K;
            int32_t *oi = idx + ((size_t)b * P1 + qi) * K;
#pragma unroll
            for (int s = 0; s < KB; ++s) {
                const int k = s - (KB - K);
                if (k >= 0) {
                    od[k] = k < L2 ? ld[r][s] : 0.0f;
                    oi[k] = k < L2 ? lj[r][s] : 0;
                }
            }
        } else {
            uint2 *o = part + (((size_t)b * n_split + blockIdx.y) * P1 + qi) * K;
#pragma unroll
            for (int s = 0; s < KB; ++s) {
                const int k = s - (KB - K);
                if (k >= 0) o[k] = make_uint2(__float_as_uint(ld[r][s]), (unsigned int)lj[r][s]);
            }
        }
    }
}

// grid = (ceil(P1 / 128), B): merge the sorted lists of the splits that hold targets of the pair (lexicographic on
// (dist, idx); the ranges are disjoint) and apply the zero fill.
__device__ __forceinline__ bool knn_before(float da, int ja, float db, int jb) {
    return da < db || (da == db && ja < jb);
}

__global__ void __launch_bounds__(128)
knn_merge_kernel(const uint2 *__restrict__ part, const int64_t *__restrict__ len1, const int64_t *__restrict__ len2,
                 int P1, int P2, int K, int split_len, int n_split, float *__restrict__ dist,
                 int32_t *__restrict__ idx) {
    pdl_wait();
    const int b = blockIdx.y;
    const int i = blockIdx.x * 128 + threadIdx.x;
    if (i >= P1) return;
    const int L1 = pair_len(len1, b, P1), L2 = pair_len(len2, b, P2);
    float *od = dist + ((size_t)b * P1 + i) * K;
    int32_t *oi = idx + ((size_t)b * P1 + i) * K;
    if (i >= L1 || L2 == 0) {
        for (int k = 0; k < K; ++k) {
            od[k] = 0.0f;
            oi[k] = 0;
        }
        return;
    }
    const int ns = (L2 + split_len - 1) / split_len;  // splits with targets of this pair (<= n_split)
    const uint2 *src = part + ((size_t)b * n_split * P1 + i) * K;
    const size_t sstride = (size_t)P1 * K;
    float hd[KNN_MAX_SPLIT];
    int hj[KNN_MAX_SPLIT], pos[KNN_MAX_SPLIT];
#pragma unroll
    for (int s = 0; s < KNN_MAX_SPLIT; ++s) {
        pos[s] = 0;
        hd[s] = __int_as_float(0x7f800000);
        hj[s] = 0x7fffffff;  // after every real slot and every (+inf, 0) placeholder
        if (s < ns) {
            const uint2 v = src[s * sstride];
            hd[s] = __uint_as_float(v.x);
            hj[s] = (int)v.y;
        }
    }
    for (int k = 0; k < K; ++k) {
        float d = hd[0];
        int j = hj[0], bs = 0;
#pragma unroll
        for (int s = 1; s < KNN_MAX_SPLIT; ++s)
            if (knn_before(hd[s], hj[s], d, j)) {
                d = hd[s];
                j = hj[s];
                bs = s;
            }
#pragma unroll
        for (int s = 0; s < KNN_MAX_SPLIT; ++s)
            if (s == bs) {
                if (++pos[s] < K) {
                    const uint2 v = src[s * sstride + pos[s]];
                    hd[s] = __uint_as_float(v.x);
                    hj[s] = (int)v.y;
                } else {
                    hd[s] = __int_as_float(0x7f800000);
                    hj[s] = 0x7fffffff;
                }
            }
        od[k] = k < L2 ? d : 0.0f;
        oi[k] = k < L2 ? j : 0;
    }
}

// ---------------------------------------------------------------------------------------- backward
// The gradient of dist[b,i,k] = |p1_i - p2_j|^2, j = idx[b,i,k], under the upstream gradient g[b,i,k].  A slot
// k < min(K, l2) of a valid query i < l1 has the term s * (p1_i - p2_j) per component, s = 2 g[b,i,k] (PyTorch3D's
// knn_points_backward); no other slot exists and its g is never read.  The 1-NN backward (ptk_knn1_bwd_*) is this code
// at K = 1.
__device__ __forceinline__ bool knn_term(const float *__restrict__ p1b, const float *__restrict__ p2b,
                                         const int32_t *__restrict__ idx, const float *__restrict__ g, int i, int k,
                                         int K, int L1, int L2, int &j, float t[3]) {
    if (i >= L1 || k >= L2) return false;
    j = idx[(size_t)i * K + k];
    const float s = 2.0f * g[(size_t)i * K + k];
    t[0] = s * (p1b[i * 3 + 0] - p2b[j * 3 + 0]);
    t[1] = s * (p1b[i * 3 + 1] - p2b[j * 3 + 1]);
    t[2] = s * (p1b[i * 3 + 2] - p2b[j * 3 + 2]);
    return true;
}

// grad_p1 row i: the terms of its slots summed in slot order, ((t0 + t1) + t2) + ..., or +0 without a term
__device__ __forceinline__ void knn_grad_p1_row(const float *__restrict__ p1b, const float *__restrict__ p2b,
                                                const int32_t *__restrict__ idx, const float *__restrict__ g, int i, int K,
                                                int L1, int L2, float *__restrict__ o) {
    float a[3] = {0.0f, 0.0f, 0.0f}, t[3];
    int j;
    for (int k = 0; k < K; ++k) {
        if (!knn_term(p1b, p2b, idx, g, i, k, K, L1, L2, j, t)) break;
        if (k == 0) {
            a[0] = t[0];
            a[1] = t[1];
            a[2] = t[2];
        } else {
            a[0] += t[0];
            a[1] += t[1];
            a[2] += t[2];
        }
    }
    o[0] = a[0];
    o[1] = a[1];
    o[2] = a[2];
}

// phase A, grid = (ceil(max(P1,P2) / 256), B): grad_p1 rows, grad_p2 rows zeroed for phase B
__global__ void __launch_bounds__(256)
knn_bwd_direct_kernel(const float *__restrict__ p1, const float *__restrict__ p2, const int32_t *__restrict__ idx,
                      const float *__restrict__ grad_dist, int P1, int P2, int K, const int64_t *__restrict__ len1,
                      const int64_t *__restrict__ len2, float *__restrict__ grad_p1, float *__restrict__ grad_p2) {
    pdl_wait();
    const int b = blockIdx.y;
    const int i = blockIdx.x * 256 + threadIdx.x;
    const int L1 = pair_len(len1, b, P1), L2 = pair_len(len2, b, P2);
    if (grad_p1 && i < P1)
        knn_grad_p1_row(p1 + (size_t)b * P1 * 3, p2 + (size_t)b * P2 * 3, idx + (size_t)b * P1 * K,
                        grad_dist + (size_t)b * P1 * K, i, K, L1, L2, grad_p1 + ((size_t)b * P1 + i) * 3);
    if (grad_p2 && i < P2) {
        float *o = grad_p2 + ((size_t)b * P2 + i) * 3;
        o[0] = o[1] = o[2] = 0.0f;
    }
}

// phase B, grid = (ceil(P1 * K / 256), B), one thread per slot: grad_p2[b, j] -= term, RED.ADD.F32
__global__ void __launch_bounds__(256)
knn_bwd_scatter_kernel(const float *__restrict__ p1, const float *__restrict__ p2, const int32_t *__restrict__ idx,
                       const float *__restrict__ grad_dist, int P1, int P2, int K, const int64_t *__restrict__ len1,
                       const int64_t *__restrict__ len2, float *__restrict__ grad_p2) {
    pdl_wait();
    const int b = blockIdx.y;
    const int e = blockIdx.x * 256 + threadIdx.x;
    if (e >= P1 * K) return;
    const int L1 = pair_len(len1, b, P1), L2 = pair_len(len2, b, P2);
    float t[3];
    int j;
    if (knn_term(p1 + (size_t)b * P1 * 3, p2 + (size_t)b * P2 * 3, idx + (size_t)b * P1 * K,
                 grad_dist + (size_t)b * P1 * K, e / K, e % K, K, L1, L2, j, t)) {
        float *o = grad_p2 + ((size_t)b * P2 + j) * 3;
        atomicAdd(o + 0, -t[0]);
        atomicAdd(o + 1, -t[1]);
        atomicAdd(o + 2, -t[2]);
    }
}

// Deterministic form (det_accum.cuh): grad_p1 is phase A's slot-order sum; grad_p2 goes through the integer sum with
// M_b = the largest finite |term| of pair b and n = l1 + 1 (a query's K indices are distinct, so a p2 row receives at
// most l1 terms).
// phase 1, grid = (ceil(max(P1 * K, P2) / 256), B): M_b over the slots (atomicMax into mbits[b], zeroed by the
// caller), grad_p1 rows as in phase A, accumulators and outputs of every p2 row zeroed
__global__ void __launch_bounds__(256)
knn_bwd_det_terms_kernel(const float *__restrict__ p1, const float *__restrict__ p2, const int32_t *__restrict__ idx,
                         const float *__restrict__ grad_dist, int P1, int P2, int K, const int64_t *__restrict__ len1,
                         const int64_t *__restrict__ len2, float *__restrict__ grad_p1, float *__restrict__ grad_p2,
                         unsigned long long *__restrict__ acc, unsigned int *__restrict__ mbits) {
    pdl_wait();
    const int b = blockIdx.y;
    const int e = blockIdx.x * 256 + threadIdx.x;
    const int L1 = pair_len(len1, b, P1), L2 = pair_len(len2, b, P2);
    const float *p1b = p1 + (size_t)b * P1 * 3, *p2b = p2 + (size_t)b * P2 * 3;
    const int32_t *ib = idx + (size_t)b * P1 * K;
    const float *gb = grad_dist + (size_t)b * P1 * K;
    float m = 0.0f, t[3];
    int j;
    if (e < P1 * K && knn_term(p1b, p2b, ib, gb, e / K, e % K, K, L1, L2, j, t))
        m = fmaxf(det_abs_finite(t[0]), fmaxf(det_abs_finite(t[1]), det_abs_finite(t[2])));
    if (grad_p1 && e < P1) knn_grad_p1_row(p1b, p2b, ib, gb, e, K, L1, L2, grad_p1 + ((size_t)b * P1 + e) * 3);
    if (e < P2) det_zero_row(acc, grad_p2, (size_t)b * P2 + e);
    det_block_max<256>(m, mbits + b);
}

// phase 2, grid = (ceil(P1 * K / 256), B): quantise and add into the neighbour's row (non-finite terms into grad_p2)
__global__ void __launch_bounds__(256)
knn_bwd_det_reduce_kernel(const float *__restrict__ p1, const float *__restrict__ p2, const int32_t *__restrict__ idx,
                          const float *__restrict__ grad_dist, int P1, int P2, int K, const int64_t *__restrict__ len1,
                          const int64_t *__restrict__ len2, float *__restrict__ grad_p2,
                          unsigned long long *__restrict__ acc, const unsigned int *__restrict__ mbits, DetBound nb) {
    pdl_wait();
    const int b = blockIdx.y;
    const int e = blockIdx.x * 256 + threadIdx.x;
    if (e >= P1 * K) return;
    const int L1 = pair_len(len1, b, P1), L2 = pair_len(len2, b, P2);
    float t[3];
    int j;
    if (!knn_term(p1 + (size_t)b * P1 * 3, p2 + (size_t)b * P2 * 3, idx + (size_t)b * P1 * K,
                  grad_dist + (size_t)b * P1 * K, e / K, e % K, K, L1, L2, j, t))
        return;
    const double scale = det_scale(mbits, nb, b);
    const size_t r = ((size_t)b * P2 + j) * 3;
#pragma unroll
    for (int d = 0; d < 3; ++d) det_add(acc + r + d, grad_p2 + r + d, -t[d], scale);
}

// ---------------------------------------------------------------------------------------- host side
struct KnnPlan {
    int n_split;    // CTAs along the target range
    int split_len;  // targets per split (a multiple of KNN_CHUNK)
};

// A pure function of the shapes, so that the workspace size is one too: split the target range while the query
// blocks alone give fewer than KNN_FILL_CTAS CTAs, into at most KNN_MAX_SPLIT ranges of at least KNN_MIN_SPLIT_LEN.
static KnnPlan knn_plan(int64_t B, int64_t P1, int64_t P2, int K) {
    const int64_t base = B * ceil_div(P1, (int64_t)KNN_THREADS * knn_rows(knn_bucket(K)));
    int64_t ns = base >= KNN_FILL_CTAS ? 1 : ceil_div(KNN_FILL_CTAS, base);
    ns = std::min<int64_t>(ns, std::min<int64_t>(KNN_MAX_SPLIT, ceil_div(P2, (int64_t)KNN_MIN_SPLIT_LEN)));
    ns = std::max<int64_t>(ns, 1);
    KnnPlan p;
    const int64_t len = ceil_div(ceil_div(P2, ns), (int64_t)KNN_CHUNK) * KNN_CHUNK;
    p.n_split = (int)ceil_div(P2, len);
    p.split_len = (int)len;
    return p;
}

static int check_knn(const float *p1, const float *p2, int64_t B, int64_t P1, int64_t P2, int64_t K) {
    int rc = check_clouds(p1, p2, B, P1, P2);
    if (rc) return rc;
    PTK_REQUIRE(K >= 1 && K <= PTK_KNN_MAX_K, PTK_ERR_SHAPE, "knn: K=%lld outside [1, %d]", (long long)K,
                PTK_KNN_MAX_K);
    PTK_REQUIRE(B <= 65535, PTK_ERR_SHAPE, "knn: batch too large");
    PTK_REQUIRE(P1 * K < (1LL << 31), PTK_ERR_SHAPE, "knn: P1 * K too large for 32-bit indexing");
    return PTK_OK;
}

extern "C" size_t ptk_knn_workspace_bytes(int64_t B, int64_t P1, int64_t P2, int64_t K) {
    if (B <= 0 || P1 <= 0 || P2 <= 0 || K < 1 || K > PTK_KNN_MAX_K) return 0;
    const KnnPlan p = knn_plan(B, P1, P2, (int)K);
    return p.n_split > 1 ? (size_t)B * p.n_split * (size_t)P1 * (size_t)K * sizeof(uint2) : 0;
}

template <int KB>
static void launch_knn_scan(dim3 grid, cudaStream_t st, const float *p1, const float *p2, const int64_t *len1,
                            const int64_t *len2, int P1, int P2, int K, const KnnPlan &p, float *dist, int32_t *idx,
                            uint2 *part) {
    launch_pdl(knn_scan_kernel<KB, knn_rows(KB), knn_minb(KB)>, grid, dim3(KNN_THREADS), 0, st, p1, p2, len1, len2, P1,
               P2, K, p.split_len, p.n_split, dist, idx, part);
}

extern "C" int ptk_knn_fwd_lengths(const float *p1, const float *p2, const int64_t *len1, const int64_t *len2, int64_t B,
                                   int64_t P1, int64_t P2, int64_t K, float *dist, int32_t *idx, void *workspace,
                                   size_t workspace_bytes, ptk_stream_t stream) {
    PTK_NVTX("ptk_knn_fwd_lengths");
    int rc = check_knn(p1, p2, B, P1, P2, K);
    if (rc) return rc;
    PTK_REQUIRE(dist && idx, PTK_ERR_SHAPE, "knn_fwd: null dist / idx pointer");
    const size_t need = ptk_knn_workspace_bytes(B, P1, P2, K);
    PTK_REQUIRE(workspace_bytes >= need && (need == 0 || workspace), PTK_ERR_WORKSPACE,
                "knn_fwd: workspace too small (%zu < %zu)", workspace_bytes, need);
    PTK_REQUIRE((reinterpret_cast<uintptr_t>(workspace) & 15) == 0, PTK_ERR_ALIGN,
                "knn_fwd: workspace must be 16-byte aligned");
    cudaStream_t st = as_stream(stream);
    const KnnPlan p = knn_plan(B, P1, P2, (int)K);
    const int KB = knn_bucket((int)K);
    const dim3 grid((unsigned)ceil_div(P1, (int64_t)KNN_THREADS * knn_rows(KB)), (unsigned)p.n_split, (unsigned)B);
    uint2 *part = p.n_split > 1 ? reinterpret_cast<uint2 *>(workspace) : nullptr;
    const int iP1 = (int)P1, iP2 = (int)P2, iK = (int)K;
    switch (KB) {
        case 2: launch_knn_scan<2>(grid, st, p1, p2, len1, len2, iP1, iP2, iK, p, dist, idx, part); break;
        case 4: launch_knn_scan<4>(grid, st, p1, p2, len1, len2, iP1, iP2, iK, p, dist, idx, part); break;
        case 8: launch_knn_scan<8>(grid, st, p1, p2, len1, len2, iP1, iP2, iK, p, dist, idx, part); break;
        case 16: launch_knn_scan<16>(grid, st, p1, p2, len1, len2, iP1, iP2, iK, p, dist, idx, part); break;
        case 32: launch_knn_scan<32>(grid, st, p1, p2, len1, len2, iP1, iP2, iK, p, dist, idx, part); break;
        default: launch_knn_scan<64>(grid, st, p1, p2, len1, len2, iP1, iP2, iK, p, dist, idx, part); break;
    }
    PTK_CHECK_LAUNCH();
    if (p.n_split > 1) {
        launch_pdl(knn_merge_kernel, dim3((unsigned)ceil_div(P1, (int64_t)128), (unsigned)B), dim3(128), 0, st,
                   (const uint2 *)part, len1, len2, iP1, iP2, iK, p.split_len, p.n_split, dist, idx);
        PTK_CHECK_LAUNCH();
    }
    return PTK_OK;
}

// The backward bodies behind ptk_knn_bwd_* and ptk_knn1_bwd_* (K = 1); the caller has checked the arguments and that
// a gradient is requested.
static int knn_bwd(const float *p1, const float *p2, const int64_t *len1, const int64_t *len2, const int32_t *idx,
                   const float *grad_dist, int64_t B, int64_t P1, int64_t P2, int64_t K, float *grad_p1, float *grad_p2,
                   cudaStream_t st) {
    const int64_t Pm = P1 > P2 ? P1 : P2;
    launch_pdl(knn_bwd_direct_kernel, dim3((unsigned)ceil_div(Pm, 256), (unsigned)B), dim3(256), 0, st, p1, p2, idx,
               grad_dist, (int)P1, (int)P2, (int)K, len1, len2, grad_p1, grad_p2);
    PTK_CHECK_LAUNCH();
    if (grad_p2) {
        launch_pdl(knn_bwd_scatter_kernel, dim3((unsigned)ceil_div(P1 * K, 256), (unsigned)B), dim3(256), 0, st, p1, p2,
                   idx, grad_dist, (int)P1, (int)P2, (int)K, len1, len2, grad_p2);
        PTK_CHECK_LAUNCH();
    }
    return PTK_OK;
}

// workspace: det_workspace_bytes(B, P2), checked by the caller
static int knn_bwd_det(const float *p1, const float *p2, const int64_t *len1, const int64_t *len2, const int32_t *idx,
                       const float *grad_dist, int64_t B, int64_t P1, int64_t P2, int64_t K, float *grad_p1,
                       float *grad_p2, void *workspace, cudaStream_t st) {
    if (!grad_p2) return knn_bwd(p1, p2, len1, len2, idx, grad_dist, B, P1, P2, K, grad_p1, nullptr, st);  // plain stores
    DetWs w;
    PTK_CHECK_CUDA(det_begin(workspace, B, P2, st, w));
    const DetBound nb = det_bound_len(len1, P1);
    const int64_t PK = P1 * K > P2 ? P1 * K : P2;
    launch_pdl(knn_bwd_det_terms_kernel, dim3((unsigned)ceil_div(PK, 256), (unsigned)B), dim3(256), 0, st, p1, p2, idx,
               grad_dist, (int)P1, (int)P2, (int)K, len1, len2, grad_p1, grad_p2, w.acc_a, w.mbits);
    PTK_CHECK_LAUNCH();
    launch_pdl(knn_bwd_det_reduce_kernel, dim3((unsigned)ceil_div(P1 * K, 256), (unsigned)B), dim3(256), 0, st, p1, p2,
               idx, grad_dist, (int)P1, (int)P2, (int)K, len1, len2, grad_p2, w.acc_a, (const unsigned int *)w.mbits, nb);
    PTK_CHECK_LAUNCH();
    det_launch_convert<256>(w, nb, B, grad_p2, P2, nullptr, 0, st);
    PTK_CHECK_LAUNCH();
    return PTK_OK;
}

static int knn_bwd_check(const float *p1, const float *p2, const int32_t *idx, const float *grad_dist, int64_t B,
                         int64_t P1, int64_t P2, int64_t K) {
    int rc = check_knn(p1, p2, B, P1, P2, K);
    if (rc) return rc;
    PTK_REQUIRE(idx && grad_dist, PTK_ERR_SHAPE, "knn_bwd: null index / grad pointer");
    return PTK_OK;
}

}  // namespace ptk

using namespace ptk;

extern "C" int ptk_knn_bwd_lengths(const float *p1, const float *p2, const int64_t *len1, const int64_t *len2,
                                   const int32_t *idx, const float *grad_dist, int64_t B, int64_t P1, int64_t P2,
                                   int64_t K, float *grad_p1, float *grad_p2, ptk_stream_t stream) {
    PTK_NVTX("ptk_knn_bwd_lengths");
    int rc = knn_bwd_check(p1, p2, idx, grad_dist, B, P1, P2, K);
    if (rc) return rc;
    if (!grad_p1 && !grad_p2) return PTK_OK;
    return knn_bwd(p1, p2, len1, len2, idx, grad_dist, B, P1, P2, K, grad_p1, grad_p2, as_stream(stream));
}

extern "C" size_t ptk_knn1_bwd_det_workspace_bytes(int64_t B, int64_t P1, int64_t P2) {
    if (B <= 0 || P1 <= 0 || P2 <= 0) return 0;
    return det_workspace_bytes(B, P2);
}

extern "C" int ptk_knn_bwd_det(const float *p1, const float *p2, const int64_t *len1, const int64_t *len2,
                               const int32_t *idx, const float *grad_dist, int64_t B, int64_t P1, int64_t P2, int64_t K,
                               float *grad_p1, float *grad_p2, void *workspace, size_t workspace_bytes,
                               ptk_stream_t stream) {
    PTK_NVTX("ptk_knn_bwd_det");
    int rc = knn_bwd_check(p1, p2, idx, grad_dist, B, P1, P2, K);
    if (rc) return rc;
    if (!grad_p1 && !grad_p2) return PTK_OK;
    rc = det_check_workspace(workspace, workspace_bytes, ptk_knn1_bwd_det_workspace_bytes(B, P1, P2), "knn_bwd_det");
    if (rc) return rc;
    return knn_bwd_det(p1, p2, len1, len2, idx, grad_dist, B, P1, P2, K, grad_p1, grad_p2, workspace, as_stream(stream));
}

static int knn1_bwd_check(const float *p1, const float *p2, const int32_t *idx, const float *grad_dist, int64_t B,
                          int64_t P1, int64_t P2) {
    int rc = check_clouds(p1, p2, B, P1, P2);
    if (rc) return rc;
    PTK_REQUIRE(idx && grad_dist, PTK_ERR_SHAPE, "knn1_bwd: null index / grad pointer");
    return PTK_OK;
}

extern "C" int ptk_knn1_bwd_lengths(const float *p1, const float *p2, const int64_t *len1, const int64_t *len2,
                                    const int32_t *idx, const float *grad_dist, int64_t B, int64_t P1, int64_t P2,
                                    float *grad_p1, float *grad_p2, ptk_stream_t stream) {
    PTK_NVTX("ptk_knn1_bwd_lengths");
    int rc = knn1_bwd_check(p1, p2, idx, grad_dist, B, P1, P2);
    if (rc) return rc;
    if (!grad_p1 && !grad_p2) return PTK_OK;
    PTK_REQUIRE(B <= 65535, PTK_ERR_SHAPE, "knn1_bwd: batch too large");
    return knn_bwd(p1, p2, len1, len2, idx, grad_dist, B, P1, P2, 1, grad_p1, grad_p2, as_stream(stream));
}

extern "C" int ptk_knn1_bwd_det(const float *p1, const float *p2, const int64_t *len1, const int64_t *len2,
                                const int32_t *idx, const float *grad_dist, int64_t B, int64_t P1, int64_t P2,
                                float *grad_p1, float *grad_p2, void *workspace, size_t workspace_bytes,
                                ptk_stream_t stream) {
    PTK_NVTX("ptk_knn1_bwd_det");
    int rc = knn1_bwd_check(p1, p2, idx, grad_dist, B, P1, P2);
    if (rc) return rc;
    if (!grad_p1 && !grad_p2) return PTK_OK;
    rc = det_check_workspace(workspace, workspace_bytes, ptk_knn1_bwd_det_workspace_bytes(B, P1, P2), "knn1_bwd_det");
    if (rc) return rc;
    PTK_REQUIRE(B <= 65535, PTK_ERR_SHAPE, "knn1_bwd_det: batch too large");
    return knn_bwd_det(p1, p2, len1, len2, idx, grad_dist, B, P1, P2, 1, grad_p1, grad_p2, workspace, as_stream(stream));
}
