// Pruned exact 1-NN scan (PTK_CHAMFER_PRUNED): the brute-force contract's results -- bit-identical distances,
// lowest index on exact ties -- without evaluating every (query, target) pair.  SURVEY.md 8f N4 lists a spatial
// structure for the >= 50k-point clouds of BASELINE config 5 as the optional next step; this is it.
//
//   chamfer_pruned_sort_kernel    one CTA per cloud: bounding box, G^3 cells ranked along a Hilbert curve, counting sort (shared-memory
//                                 histogram), the cloud rewritten in cell order as 16-point leaf chunks
//                                 [x16 | y16 | z16 | original index16] (256 B, two cache lines per chunk), and a
//                                 3-level box hierarchy over the chunks (fan-out 32): leaf chunk, 512 points, 16k points.
//   chamfer_pruned_query_kernel   one warp per 32 consecutive SORTED queries (a compact patch of the query cloud).
//                                 Box tests run lane-parallel (lane = child box) against the warp's query box and
//                                 are visited best-first (redux.sync min over the lower bounds), so the nearest leaf
//                                 is scanned first and a level stops as soon as its smallest remaining bound exceeds
//                                 the largest current best of the warp.  A surviving leaf is tested per query and
//                                 then scanned by all 32 lanes with uniform (broadcast) 128-bit loads and the packed
//                                 FP32x2 defining arithmetic: 68 instructions per 512 evaluations.
//
// Why it is exact.  A box bound is  lb = fma(gz,gz, fma(gy,gy, gx*gx))  with  g = max(lo - q_hi, q_lo - hi, 0)  per axis,
// the SAME operation sequence as the distance  d = fma(dz,dz, fma(dy,dy, dx*dx)),  dx = q - t.  For a target inside the
// box, rounding is monotone: fl(t - q) >= fl(lo - q_hi) > 0 when the box lies above the query (symmetrically below), so
// g <= |dx| holds for the COMPUTED values, squares and FMAs of non-negative operands preserve the order, and therefore
// lb <= d as computed -- no epsilon.  A box is skipped only when lb > best (strictly), so no target that could beat
// or tie the incumbent is ever skipped.  Sorted order is not index order, so a query keeps the pair (best distance,
// lowest ORIGINAL index attaining it) and a scanned leaf updates it lexicographically: when any query of the warp
// improves or ties, the leaf's 16 original indices are loaded (uniform) and the lowest one among the leaf's exact
// minima competes -- PyTorch3D's "lowest index wins ties" without any dependence on the visiting order.
// Every query of a cloud pair with non-finite (or overflow-prone) coordinates, and of a warp that had to scan more than
// an eighth of all leaves (strongly clustered clouds defeat a uniform grid), is appended to the rescue list and re-scanned by chamfer_nn_exact2_kernel in list mode, as the
// filter path does with its ambiguous queries.  The order of points inside a cell depends on the scheduling of
// shared-memory atomics; results do not (a (distance, lowest original index) minimum is order-free).
#pragma once
#include "chamfer_kernel2.cuh"

namespace ptk {

constexpr int PR_CHUNK = 16;  // targets per leaf
constexpr int PR_FAN = 32;    // children per inner node (= lanes of the box test)
constexpr int PR_SORT_THREADS = 1024;
constexpr int PR_QUERY_WARPS = 4;  // small CTAs: a slot frees as soon as its 4 patches are done
constexpr int PR_MAX_POINTS = PR_CHUNK * PR_FAN * PR_FAN * PR_FAN;  // 524288: one top-level group of 32 boxes

#ifdef PTK_PR_STATS
// development counters: [0] warps, [1] level-2 pops, [2] level-1 pops, [3] leaf pops (per-query tests), [4] leaf scans, [5] bails
__device__ unsigned long long pr_stats[16];  // [8..15]: sort-kernel phase cycles (thread 0 of every CTA)
#define PR_PHASE(i) do { if (threadIdx.x == 0) { const long long t_ = clock64(); atomicAdd(&pr_stats[8 + (i)], (unsigned long long)(t_ - t_phase)); t_phase = t_; } } while (0)
#define PR_STAT(i, n) do { if (lane == 0) atomicAdd(&pr_stats[i], (unsigned long long)(n)); } while (0)
#else
#define PR_STAT(i, n) do { } while (0)
#define PR_PHASE(i) do { } while (0)
#endif

struct PrBox {
    float4 lo, hi;  // .xyz; .w unused
};

__host__ __device__ inline int pr_nb0(int P) { return (P + PR_CHUNK - 1) / PR_CHUNK; }
__host__ __device__ inline int pr_nb1(int P) { return (pr_nb0(P) + PR_FAN - 1) / PR_FAN; }
__host__ __device__ inline int pr_nb2(int P) { return (pr_nb1(P) + PR_FAN - 1) / PR_FAN; }
__host__ __device__ inline int pr_boxes(int P) { return pr_nb0(P) + pr_nb1(P) + pr_nb2(P); }

// Cell order: position of cell (cx, cy, cz) along the 3-D Hilbert curve of a 2^BITS grid (Skilling's axes-to-transpose
// transform, "Programming the Hilbert curve", AIP Conf. Proc. 707, 2004, followed by the bit interleave).  Unlike the
// Morton (Z) order, consecutive cells are always face neighbours: a leaf of 16 consecutive points, and a warp's 32
// consecutive queries, never straddle a jump of the curve, so their boxes stay compact (with the Z order the few
// patches that straddled a jump had boxes as large as the cloud and dominated the tail of the query kernel).
template <int BITS>
__device__ __forceinline__ unsigned pr_cell_rank(int cx, int cy, int cz) {
    unsigned X0 = (unsigned)cx, X1 = (unsigned)cy, X2 = (unsigned)cz;
#pragma unroll
    for (unsigned Q = 1u << (BITS - 1); Q > 1; Q >>= 1) {
        const unsigned Pm = Q - 1;
        unsigned t;
        if (X0 & Q) X0 ^= Pm;  // (the exchange of X0 with itself is the identity)
        if (X1 & Q) X0 ^= Pm; else { t = (X0 ^ X1) & Pm; X0 ^= t; X1 ^= t; }
        if (X2 & Q) X0 ^= Pm; else { t = (X0 ^ X2) & Pm; X0 ^= t; X2 ^= t; }
    }
    X1 ^= X0;
    X2 ^= X1;
    unsigned t = 0;
#pragma unroll
    for (unsigned Q = 1u << (BITS - 1); Q > 1; Q >>= 1)
        if (X2 & Q) t ^= Q - 1;
    X0 ^= t, X1 ^= t, X2 ^= t;
    unsigned code = 0;
#pragma unroll
    for (int k = 0; k < BITS; ++k)
        code |= ((X2 >> k) & 1u) << (3 * k) | ((X1 >> k) & 1u) << (3 * k + 1) | ((X0 >> k) & 1u) << (3 * k + 2);
    return code;
}

// grid = 2 * B (blockIdx.x = 2 * b + cloud), block = 1024, dynamic shared memory = 4 * 8^BITS bytes (the histogram)
// + 2 * max(P1, P2) bytes when keep_codes.
template <int BITS>
__global__ void __launch_bounds__(PR_SORT_THREADS)
chamfer_pruned_sort_kernel(const float *__restrict__ x, const float *__restrict__ y, int P1, int P2,
                           const int64_t *__restrict__ len_x, const int64_t *__restrict__ len_y, float *soa_x,
                           float *soa_y, float4 *stage_x, float4 *stage_y, PrBox *box_x, PrBox *box_y,
                           int *__restrict__ bad_flags, unsigned int *__restrict__ rescue_count, int keep_codes) {
    constexpr int G = 1 << BITS, NC = G * G * G, PER = NC / PR_SORT_THREADS;
    static_assert(NC % PR_SORT_THREADS == 0, "histogram must split evenly over the threads");
    extern __shared__ unsigned int pr_hist[];
    __shared__ float sred[6][32];
    __shared__ float sbox[6];
    __shared__ unsigned int swsum[32];
    __shared__ int sbad;
    pdl_wait();
    long long t_phase = clock64();
    (void)t_phase;
    const int b = blockIdx.x >> 1, cloud = blockIdx.x & 1;
    const int tid = threadIdx.x;
    // Pc sizes the layout (padded cloud); only the cloud's first P points exist and are sorted.  Leaves past them hold
    // padding only: their box is empty (lo = +inf, hi = -inf), its lower bound +inf, and so is that of an inner box
    // over such leaves -- never below a live query's best once one leaf has been scanned.
    const int Pc = cloud == 0 ? P1 : P2;
    const int P = pair_len(cloud == 0 ? len_x : len_y, b, Pc);
    const int Pp = soa_padded(Pc);
    const float *__restrict__ src = cloud == 0 ? x + (size_t)b * P1 * 3 : y + (size_t)b * P2 * 3;
    float *out = cloud == 0 ? soa_x + (size_t)b * 4 * Pp : soa_y + (size_t)b * 4 * Pp;
    float4 *stage = cloud == 0 ? stage_x + (size_t)b * Pp : stage_y + (size_t)b * Pp;
    PrBox *box0 = (cloud == 0 ? box_x : box_y) + (size_t)b * pr_boxes(Pc);
    const int nb0 = pr_nb0(Pc), nb1 = pr_nb1(Pc), nb2 = pr_nb2(Pc);
    PrBox *box1 = box0 + nb0, *box2 = box1 + nb1;
    const float PINF = __int_as_float(0x7f800000), NINF = __int_as_float(0xff800000);
    if (tid == 0) sbad = 0;
    for (int c = tid; c < NC; c += PR_SORT_THREADS) pr_hist[c] = 0u;

    // ---- bounding box (thread t reads elements t, t + 1024, ...: coordinate index advances by 1024 % 3 == 1)
    float lo[3] = {PINF, PINF, PINF}, hi[3] = {NINF, NINF, NINF};
    bool bad = false;
    {
        const int n = P * 3;
        for (int e0 = tid; e0 < n; e0 += 8 * PR_SORT_THREADS) {
            float v[8];
#pragma unroll
            for (int u = 0; u < 8; ++u) v[u] = e0 + u * PR_SORT_THREADS < n ? src[e0 + u * PR_SORT_THREADS] : src[tid % 3];
#pragma unroll
            for (int u = 0; u < 8; ++u) {
                const int e = e0 + u * PR_SORT_THREADS < n ? e0 + u * PR_SORT_THREADS : tid % 3;
                const int c = e % 3;
                bad |= !(fabsf(v[u]) <= 1.0e15f);  // NaN, Inf, or squares that could overflow
#pragma unroll
                for (int k = 0; k < 3; ++k)
                    if (k == c) {
                        lo[k] = fminf(lo[k], v[u]);
                        hi[k] = fmaxf(hi[k], v[u]);
                    }
            }
        }
    }
    __syncthreads();
    if (bad) sbad = 1;
#pragma unroll
    for (int c = 0; c < 3; ++c) {
        float l = lo[c], h = hi[c];
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            l = fminf(l, __shfl_xor_sync(0xffffffffu, l, o));
            h = fmaxf(h, __shfl_xor_sync(0xffffffffu, h, o));
        }
        if ((tid & 31) == 0) {
            sred[c][tid >> 5] = l;
            sred[3 + c][tid >> 5] = h;
        }
    }
    __syncthreads();
    if (tid < 3) {
        float l = sred[tid][0], h = sred[3 + tid][0];
        for (int w = 1; w < 32; ++w) {
            l = fminf(l, sred[tid][w]);
            h = fmaxf(h, sred[3 + tid][w]);
        }
        sbox[tid] = l;
        sbox[3 + tid] = h;
    }
    __syncthreads();
    PR_PHASE(0);  // bounding box
    const bool cloud_bad = sbad != 0;
    float org[3], scl[3];
#pragma unroll
    for (int c = 0; c < 3; ++c) {
        const float ext = sbox[3 + c] - sbox[c];
        org[c] = cloud_bad ? 0.f : sbox[c];
        scl[c] = (!cloud_bad && ext > 0.f) ? (float)G / ext : 0.f;  // a flat axis (or a bad cloud) collapses to cell 0
    }
    if (tid == 0) {
        bad_flags[2 * b + cloud] = cloud_bad ? 1 : 0;
        rescue_count[2 * b + cloud] = 0u;
    }
    auto cell_of = [&](float px, float py, float pz) {
        const int cx = min(G - 1, max(0, __float2int_rz((px - org[0]) * scl[0])));
        const int cy = min(G - 1, max(0, __float2int_rz((py - org[1]) * scl[1])));
        const int cz = min(G - 1, max(0, __float2int_rz((pz - org[2]) * scl[2])));
        return pr_cell_rank<BITS>(cx, cy, cz);
    };

    // ---- histogram over the cells; four points (twelve loads) in flight per thread.  The cell rank of a point is
    // computed once and kept as 16 bits in shared memory when the launch reserved room for it (keep_codes).
    unsigned short *codes = reinterpret_cast<unsigned short *>(pr_hist + NC);
    for (int i0 = tid; i0 < P; i0 += 4 * PR_SORT_THREADS) {
        float v[4][3];
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            const int i = min(i0 + u * PR_SORT_THREADS, P - 1);
            v[u][0] = src[3 * i], v[u][1] = src[3 * i + 1], v[u][2] = src[3 * i + 2];
        }
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            const int i = i0 + u * PR_SORT_THREADS;
            if (i < P) {
                const unsigned code = cell_of(v[u][0], v[u][1], v[u][2]);
                if (keep_codes) codes[i] = (unsigned short)code;
                atomicAdd(&pr_hist[code], 1u);
            }
        }
    }
    __syncthreads();

    PR_PHASE(1);  // histogram
    // ---- exclusive scan of the histogram (thread owns PER consecutive cells)
    {
        unsigned int sum = 0;
#pragma unroll
        for (int k = 0; k < PER; ++k) sum += pr_hist[tid * PER + k];
        unsigned int inc = sum;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const unsigned int v = __shfl_up_sync(0xffffffffu, inc, o);
            if ((tid & 31) >= o) inc += v;
        }
        if ((tid & 31) == 31) swsum[tid >> 5] = inc;
        __syncthreads();
        if (tid < 32) {
            unsigned int w = swsum[tid], winc = w;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const unsigned int v = __shfl_up_sync(0xffffffffu, winc, o);
                if (tid >= o) winc += v;
            }
            swsum[tid] = winc - w;
        }
        __syncthreads();
        unsigned int run = swsum[tid >> 5] + inc - sum;
#pragma unroll
        for (int k = 0; k < PER; ++k) {
            const unsigned int c = pr_hist[tid * PER + k];
            pr_hist[tid * PER + k] = run;
            run += c;
        }
    }
    __syncthreads();

    PR_PHASE(2);  // scan
    // ---- scatter into cell order: ONE 16-byte store per point (x, y, z, original index) into the staging array --
    // four scalar stores per point into the leaf-blocked layout cost four 32-byte sectors each and were 60 % of this
    // kernel.  The leaf pass below transposes the staged points into the layout the query kernel reads.
    for (int i0 = tid; i0 < P; i0 += 4 * PR_SORT_THREADS) {
        float v[4][3];
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            const int i = min(i0 + u * PR_SORT_THREADS, P - 1);
            v[u][0] = src[3 * i], v[u][1] = src[3 * i + 1], v[u][2] = src[3 * i + 2];
        }
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            const int i = i0 + u * PR_SORT_THREADS;
            if (i < P) {
                const unsigned code = keep_codes ? (unsigned)codes[i] : cell_of(v[u][0], v[u][1], v[u][2]);
                const unsigned int pos = atomicAdd(&pr_hist[code], 1u);
                stage[pos] = make_float4(v[u][0], v[u][1], v[u][2], __int_as_float(i));
            }
        }
    }
    __syncthreads();
    PR_PHASE(3);  // scatter

    // ---- leaves: a half-warp per leaf (lane = point) reads 256 staged bytes, writes the leaf [x16 | y16 | z16 | idx16]
    // (padding: +inf coordinates -- never a minimum, inert as a query) and reduces the leaf's box by shuffles; then a
    // warp per inner node (lane = child)
    {
        const int lane = tid & 31, hw = tid >> 4, l16 = tid & 15;
        const int nleaf_all = Pp / PR_CHUNK;  // including the all-padding leaves up to the padded cloud size
        for (int c = hw; c < nleaf_all; c += PR_SORT_THREADS / 16) {  // loop bounds are uniform per half-warp only:
            float *o = out + (size_t)c * 64;                             // shuffles below stay inside a half (xor < 16)
            const bool live = c * PR_CHUNK + l16 < P;
            float4 pt = make_float4(PINF, PINF, PINF, __int_as_float(0x7fffffff));
            if (live) pt = stage[c * PR_CHUNK + l16];
            o[l16] = pt.x;
            o[16 + l16] = pt.y;
            o[32 + l16] = pt.z;
            o[48 + l16] = pt.w;
            float l[3] = {pt.x, pt.y, pt.z}, h[3] = {live ? pt.x : NINF, live ? pt.y : NINF, live ? pt.z : NINF};
            const unsigned hmask = 0xffffu << (lane & 16);
#pragma unroll
            for (int off = 8; off > 0; off >>= 1)
#pragma unroll
                for (int k = 0; k < 3; ++k) {
                    l[k] = fminf(l[k], __shfl_xor_sync(hmask, l[k], off));
                    h[k] = fmaxf(h[k], __shfl_xor_sync(hmask, h[k], off));
                }
            if (l16 == 0 && c < nb0) {
                box0[c].lo = make_float4(l[0], l[1], l[2], 0.f);
                box0[c].hi = make_float4(h[0], h[1], h[2], 0.f);
            }
        }
        __syncthreads();
        for (int lvl = 0; lvl < 2; ++lvl) {
            const PrBox *child = lvl == 0 ? box0 : box1;
            PrBox *parent = lvl == 0 ? box1 : box2;
            const int nchild = lvl == 0 ? nb0 : nb1, nparent = lvl == 0 ? nb1 : nb2;
            for (int n = tid >> 5; n < nparent; n += PR_SORT_THREADS / 32) {
                const int c = n * PR_FAN + lane;
                float4 l = make_float4(PINF, PINF, PINF, 0.f), h = make_float4(NINF, NINF, NINF, 0.f);
                if (c < nchild) {
                    l = child[c].lo;
                    h = child[c].hi;
                }
#pragma unroll
                for (int off = 16; off > 0; off >>= 1) {
                    l.x = fminf(l.x, __shfl_xor_sync(0xffffffffu, l.x, off));
                    l.y = fminf(l.y, __shfl_xor_sync(0xffffffffu, l.y, off));
                    l.z = fminf(l.z, __shfl_xor_sync(0xffffffffu, l.z, off));
                    h.x = fmaxf(h.x, __shfl_xor_sync(0xffffffffu, h.x, off));
                    h.y = fmaxf(h.y, __shfl_xor_sync(0xffffffffu, h.y, off));
                    h.z = fmaxf(h.z, __shfl_xor_sync(0xffffffffu, h.z, off));
                }
                if (lane == 0) {
                    parent[n].lo = l;
                    parent[n].hi = h;
                }
            }
            __syncthreads();
        }
    }
    PR_PHASE(4);  // boxes
}

// ------------------------------------------------------------------------------------------------
// Wide form of the sort for FEW LARGE clouds (2 B <= 128 clouds of >= 16k points): one CTA per cloud leaves the chip
// idle (100k points: 317 us on 2 SMs), so every phase becomes its own small launch over (slices of 2048 points) x
// (clouds) and the histogram lives in global memory (L2 atomics):
//   init -> bbox (atomicMin / atomicMax on order-preserving keys) -> hist (+ cell ranks kept in the not-yet-used leaf
//   array) -> scan (one CTA per cloud) -> scatter (ATOMG with return, 16-byte staged stores) -> leaves -> inner boxes.
constexpr int PRW_THREADS = 256, PRW_PER_THREAD = 8, PRW_SLICE = PRW_THREADS * PRW_PER_THREAD;

struct PrWide {      // per-cloud state of the wide sort (global memory)
    unsigned int lo[3], nhi[3];  // bounding box as order-preserving keys: min of ord(v), min of ~ord(v)
    int bad;
    int pad;
};

__device__ __forceinline__ unsigned pr_ord(float f);
__device__ __forceinline__ float pr_unord(unsigned k);

// grid (ceil(NC / 1024), 2 * B), block 1024
__global__ void __launch_bounds__(1024)
pr_wide_init_kernel(PrWide *__restrict__ st, unsigned int *__restrict__ ghist, int NC, unsigned int *__restrict__ rescue_count) {
    pdl_wait();
    const int cl = blockIdx.y;
    const int c = blockIdx.x * 1024 + threadIdx.x;
    if (c < NC) ghist[(size_t)cl * NC + c] = 0u;
    if (c == 0) {
        PrWide w;
        w.lo[0] = w.lo[1] = w.lo[2] = w.nhi[0] = w.nhi[1] = w.nhi[2] = 0xffffffffu;
        w.bad = 0;
        w.pad = 0;
        st[cl] = w;
        rescue_count[cl] = 0u;
    }
}

// grid (ceil(Pmax / PRW_SLICE), 2 * B), block 256
__global__ void __launch_bounds__(PRW_THREADS)
pr_wide_bbox_kernel(const float *__restrict__ x, const float *__restrict__ y, int P1, int P2,
                    const int64_t *__restrict__ len_x, const int64_t *__restrict__ len_y, PrWide *__restrict__ st) {
    pdl_wait();
    const int cl = blockIdx.y, b = cl >> 1, cloud = cl & 1;
    const int P = pair_len(cloud == 0 ? len_x : len_y, b, cloud == 0 ? P1 : P2);  // valid points only
    const int e0 = blockIdx.x * PRW_SLICE * 3, e1 = min(P * 3, e0 + PRW_SLICE * 3);
    if (e0 >= e1) return;
    const float *__restrict__ src = cloud == 0 ? x + (size_t)b * P1 * 3 : y + (size_t)b * P2 * 3;
    const float PINF = __int_as_float(0x7f800000), NINF = __int_as_float(0xff800000);
    float lo[3] = {PINF, PINF, PINF}, hi[3] = {NINF, NINF, NINF};
    bool bad = false;
    // thread t reads elements e0 + t, + 256, ...: the coordinate index advances by 256 % 3 == 1 per step
    for (int e = e0 + threadIdx.x; e < e1; e += 8 * PRW_THREADS) {
        float v[8];
#pragma unroll
        for (int u = 0; u < 8; ++u) v[u] = e + u * PRW_THREADS < e1 ? src[e + u * PRW_THREADS] : src[e];
#pragma unroll
        for (int u = 0; u < 8; ++u) {
            const int c = (e + u * PRW_THREADS < e1 ? e + u * PRW_THREADS : e) % 3;
            bad |= !(fabsf(v[u]) <= 1.0e15f);
#pragma unroll
            for (int k = 0; k < 3; ++k)
                if (k == c) {
                    lo[k] = fminf(lo[k], v[u]);
                    hi[k] = fmaxf(hi[k], v[u]);
                }
        }
    }
#pragma unroll
    for (int k = 0; k < 3; ++k) {
        const unsigned l = __reduce_min_sync(0xffffffffu, pr_ord(lo[k])), h = __reduce_min_sync(0xffffffffu, ~pr_ord(hi[k]));
        if ((threadIdx.x & 31) == 0) {
            atomicMin(&st[cl].lo[k], l);
            atomicMin(&st[cl].nhi[k], h);
        }
    }
    if (__any_sync(0xffffffffu, bad) && (threadIdx.x & 31) == 0) atomicOr(&st[cl].bad, 1);
}

template <int BITS>
__device__ __forceinline__ void pr_wide_grid(const PrWide &w, float (&org)[3], float (&scl)[3]) {
#pragma unroll
    for (int c = 0; c < 3; ++c) {
        const float l = pr_unord(w.lo[c]), h = pr_unord(~w.nhi[c]);
        const float ext = h - l;
        org[c] = w.bad ? 0.f : l;
        scl[c] = (!w.bad && ext > 0.f) ? (float)(1 << BITS) / ext : 0.f;
    }
}
template <int BITS>
__device__ __forceinline__ unsigned pr_wide_cell(const float (&org)[3], const float (&scl)[3], float px, float py, float pz) {
    constexpr int G = 1 << BITS;
    const int cx = min(G - 1, max(0, __float2int_rz((px - org[0]) * scl[0])));
    const int cy = min(G - 1, max(0, __float2int_rz((py - org[1]) * scl[1])));
    const int cz = min(G - 1, max(0, __float2int_rz((pz - org[2]) * scl[2])));
    return pr_cell_rank<BITS>(cx, cy, cz);
}

// grid (ceil(Pmax / PRW_SLICE), 2 * B), block 256.  SCATTER = false: histogram + cell ranks (kept in `codes`, the
// leaf array the last phase overwrites); SCATTER = true: position from the scanned histogram, one staged 16-byte store.
template <int BITS, bool SCATTER>
__global__ void __launch_bounds__(PRW_THREADS)
pr_wide_hist_scatter_kernel(const float *__restrict__ x, const float *__restrict__ y, int P1, int P2,
                            const int64_t *__restrict__ len_x, const int64_t *__restrict__ len_y,
                            const PrWide *__restrict__ st, unsigned int *__restrict__ ghist, float *soa_x, float *soa_y,
                            float4 *__restrict__ stage_x, float4 *__restrict__ stage_y, int *__restrict__ bad_flags) {
    pdl_wait();
    constexpr int NC = 1 << (3 * BITS);
    const int cl = blockIdx.y, b = cl >> 1, cloud = cl & 1;
    const int Pc = cloud == 0 ? P1 : P2, Pp = soa_padded(Pc);  // layout; P: the points that exist
    const int P = pair_len(cloud == 0 ? len_x : len_y, b, Pc);
    const int i0 = blockIdx.x * PRW_SLICE + threadIdx.x;
    if (blockIdx.x * PRW_SLICE >= P) return;
    const float *__restrict__ src = cloud == 0 ? x + (size_t)b * P1 * 3 : y + (size_t)b * P2 * 3;
    unsigned int *codes = reinterpret_cast<unsigned int *>(cloud == 0 ? soa_x + (size_t)b * 4 * Pp : soa_y + (size_t)b * 4 * Pp);
    float4 *__restrict__ stage = cloud == 0 ? stage_x + (size_t)b * Pp : stage_y + (size_t)b * Pp;
    unsigned int *__restrict__ hist = ghist + (size_t)cl * NC;
    const PrWide w = st[cl];
    float org[3], scl[3];
    pr_wide_grid<BITS>(w, org, scl);
    if (!SCATTER && blockIdx.x == 0 && threadIdx.x == 0) bad_flags[cl] = w.bad;
    float v[PRW_PER_THREAD][3];
#pragma unroll
    for (int u = 0; u < PRW_PER_THREAD; ++u) {
        const int i = min(i0 + u * PRW_THREADS, P - 1);
        v[u][0] = src[3 * i], v[u][1] = src[3 * i + 1], v[u][2] = src[3 * i + 2];
    }
    if (!SCATTER) {
#pragma unroll
        for (int u = 0; u < PRW_PER_THREAD; ++u) {
            const int i = i0 + u * PRW_THREADS;
            if (i < P) {
                const unsigned code = pr_wide_cell<BITS>(org, scl, v[u][0], v[u][1], v[u][2]);
                codes[i] = code;
                atomicAdd(&hist[code], 1u);
            }
        }
    } else {
        unsigned int pos[PRW_PER_THREAD];
#pragma unroll
        for (int u = 0; u < PRW_PER_THREAD; ++u) {
            const int i = i0 + u * PRW_THREADS;
            pos[u] = i < P ? atomicAdd(&hist[codes[i]], 1u) : 0u;
        }
#pragma unroll
        for (int u = 0; u < PRW_PER_THREAD; ++u) {
            const int i = i0 + u * PRW_THREADS;
            if (i < P) stage[pos[u]] = make_float4(v[u][0], v[u][1], v[u][2], __int_as_float(i));
        }
    }
}

// grid 2 * B, block 1024: exclusive scan of a cloud's histogram in place
template <int BITS>
__global__ void __launch_bounds__(1024)
pr_wide_scan_kernel(unsigned int *__restrict__ ghist) {
    pdl_wait();
    constexpr int NC = 1 << (3 * BITS), PER = NC / 1024;
    __shared__ unsigned int swsum[32];
    unsigned int *__restrict__ hist = ghist + (size_t)blockIdx.x * NC;
    const int tid = threadIdx.x;
    // the thread's PER consecutive bins as 128-bit loads / stores (all issued before the first use)
    uint4 c4[PER / 4];
    uint4 *__restrict__ h4 = reinterpret_cast<uint4 *>(hist + tid * PER);
    unsigned int sum = 0;
#pragma unroll
    for (int k = 0; k < PER / 4; ++k) c4[k] = h4[k];
#pragma unroll
    for (int k = 0; k < PER / 4; ++k) sum += c4[k].x + c4[k].y + c4[k].z + c4[k].w;
    unsigned int inc = sum;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const unsigned int t = __shfl_up_sync(0xffffffffu, inc, o);
        if ((tid & 31) >= o) inc += t;
    }
    if ((tid & 31) == 31) swsum[tid >> 5] = inc;
    __syncthreads();
    if (tid < 32) {
        unsigned int wv = swsum[tid], winc = wv;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const unsigned int t = __shfl_up_sync(0xffffffffu, winc, o);
            if (tid >= o) winc += t;
        }
        swsum[tid] = winc - wv;
    }
    __syncthreads();
    unsigned int run = swsum[tid >> 5] + inc - sum;
#pragma unroll
    for (int k = 0; k < PER / 4; ++k) {
        uint4 o;
        o.x = run, run += c4[k].x;
        o.y = run, run += c4[k].y;
        o.z = run, run += c4[k].z;
        o.w = run, run += c4[k].w;
        h4[k] = o;
    }
}

// grid (ceil(leaves / 16), 2 * B), block 256: a half-warp per leaf -- transpose the staged points into the leaf layout,
// reduce the leaf box (the same pass as in chamfer_pruned_sort_kernel)
__global__ void __launch_bounds__(256)
pr_wide_leaf_kernel(int P1, int P2, const int64_t *__restrict__ len_x, const int64_t *__restrict__ len_y,
                    const float4 *__restrict__ stage_x, const float4 *__restrict__ stage_y, float *soa_x, float *soa_y,
                    PrBox *box_x, PrBox *box_y) {
    pdl_wait();
    const int cl = blockIdx.y, b = cl >> 1, cloud = cl & 1;
    const int Pc = cloud == 0 ? P1 : P2, Pp = soa_padded(Pc);  // layout; P: the points that exist
    const int P = pair_len(cloud == 0 ? len_x : len_y, b, Pc);
    const int c = blockIdx.x * 16 + (threadIdx.x >> 4), l16 = threadIdx.x & 15, lane = threadIdx.x & 31;
    if (c >= Pp / PR_CHUNK) return;  // uniform per half-warp
    const float4 *__restrict__ stage = cloud == 0 ? stage_x + (size_t)b * Pp : stage_y + (size_t)b * Pp;
    float *o = (cloud == 0 ? soa_x + (size_t)b * 4 * Pp : soa_y + (size_t)b * 4 * Pp) + (size_t)c * 64;
    PrBox *box0 = (cloud == 0 ? box_x : box_y) + (size_t)b * pr_boxes(Pc);
    const float PINF = __int_as_float(0x7f800000), NINF = __int_as_float(0xff800000);
    const bool live = c * PR_CHUNK + l16 < P;
    float4 pt = make_float4(PINF, PINF, PINF, __int_as_float(0x7fffffff));
    if (live) pt = stage[c * PR_CHUNK + l16];
    o[l16] = pt.x;
    o[16 + l16] = pt.y;
    o[32 + l16] = pt.z;
    o[48 + l16] = pt.w;
    float l[3] = {pt.x, pt.y, pt.z}, h[3] = {live ? pt.x : NINF, live ? pt.y : NINF, live ? pt.z : NINF};
    const unsigned hmask = 0xffffu << (lane & 16);
#pragma unroll
    for (int off = 8; off > 0; off >>= 1)
#pragma unroll
        for (int k = 0; k < 3; ++k) {
            l[k] = fminf(l[k], __shfl_xor_sync(hmask, l[k], off));
            h[k] = fmaxf(h[k], __shfl_xor_sync(hmask, h[k], off));
        }
    if (l16 == 0 && c < pr_nb0(Pc)) {
        box0[c].lo = make_float4(l[0], l[1], l[2], 0.f);
        box0[c].hi = make_float4(h[0], h[1], h[2], 0.f);
    }
}

// grid 2 * B, block 1024: the two inner levels (a warp per node, lane = child)
__global__ void __launch_bounds__(1024)
pr_wide_inner_kernel(int P1, int P2, PrBox *box_x, PrBox *box_y) {
    pdl_wait();
    const int cl = blockIdx.x, b = cl >> 1, cloud = cl & 1;
    const int P = cloud == 0 ? P1 : P2;
    PrBox *box0 = (cloud == 0 ? box_x : box_y) + (size_t)b * pr_boxes(P);
    const int nb0 = pr_nb0(P), nb1 = pr_nb1(P), nb2 = pr_nb2(P);
    PrBox *box1 = box0 + nb0, *box2 = box1 + nb1;
    const float PINF = __int_as_float(0x7f800000), NINF = __int_as_float(0xff800000);
    const int tid = threadIdx.x, lane = tid & 31;
    for (int lvl = 0; lvl < 2; ++lvl) {
        const PrBox *child = lvl == 0 ? box0 : box1;
        PrBox *parent = lvl == 0 ? box1 : box2;
        const int nchild = lvl == 0 ? nb0 : nb1, nparent = lvl == 0 ? nb1 : nb2;
        for (int n = tid >> 5; n < nparent; n += 32) {
            const int c = n * PR_FAN + lane;
            float4 l = make_float4(PINF, PINF, PINF, 0.f), h = make_float4(NINF, NINF, NINF, 0.f);
            if (c < nchild) {
                l = child[c].lo;
                h = child[c].hi;
            }
#pragma unroll
            for (int off = 16; off > 0; off >>= 1) {
                l.x = fminf(l.x, __shfl_xor_sync(0xffffffffu, l.x, off));
                l.y = fminf(l.y, __shfl_xor_sync(0xffffffffu, l.y, off));
                l.z = fminf(l.z, __shfl_xor_sync(0xffffffffu, l.z, off));
                h.x = fmaxf(h.x, __shfl_xor_sync(0xffffffffu, h.x, off));
                h.y = fmaxf(h.y, __shfl_xor_sync(0xffffffffu, h.y, off));
                h.z = fmaxf(h.z, __shfl_xor_sync(0xffffffffu, h.z, off));
            }
            if (lane == 0) {
                parent[n].lo = l;
                parent[n].hi = h;
            }
        }
        __syncthreads();
    }
}

__device__ __forceinline__ float pr_gap(float lo, float hi, float qlo, float qhi) {
    return fmaxf(fmaxf(__fsub_rn(lo, qhi), __fsub_rn(qlo, hi)), 0.f);
}
// lower bound of the defining distance between any point of [qlo, qhi] and any point of the box (see the header)
__device__ __forceinline__ float pr_lb(const float4 lo, const float4 hi, float qlx, float qly, float qlz, float qhx,
                                       float qhy, float qhz) {
    const float gx = pr_gap(lo.x, hi.x, qlx, qhx), gy = pr_gap(lo.y, hi.y, qly, qhy), gz = pr_gap(lo.z, hi.z, qlz, qhz);
    float d = __fmul_rn(gx, gx);
    d = __fmaf_rn(gy, gy, d);
    d = __fmaf_rn(gz, gz, d);
    return d;
}
// order-preserving map float -> unsigned (for redux.sync min / max over signed floats)
__device__ __forceinline__ unsigned pr_ord(float f) {
    const unsigned u = __float_as_uint(f);
    return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}
__device__ __forceinline__ float pr_unord(unsigned k) {
    return __uint_as_float((k & 0x80000000u) ? (k & 0x7fffffffu) : ~k);
}

// grid (ceil(max queries / (32 R x warps per CTA)), B * ndir), block = 128: a warp owns 32 R consecutive sorted queries,
// R per lane (positions base + lane, base + 32 + lane, ...).  R = 1 is what runs; R = 2 halves the loads per (query, leaf)
// pair -- the kernel is bound by the L1 return path, DESIGN.md K1b -- but its wider query box costs as much (chamfer.cu).
template <int R>
__global__ void __launch_bounds__(PR_QUERY_WARPS * 32)
chamfer_pruned_query_kernel(const float *__restrict__ soa_x, const float *__restrict__ soa_y,
                            const PrBox *__restrict__ box_x, const PrBox *__restrict__ box_y,
                            const int *__restrict__ bad_flags, int P1, int P2, const int64_t *__restrict__ len_x,
                            const int64_t *__restrict__ len_y, u64 *__restrict__ keys_x,
                            u64 *__restrict__ keys_y, int dir_only, int *__restrict__ rescue_x,
                            int *__restrict__ rescue_y, unsigned int *__restrict__ rescue_count) {
    pdl_wait();
    const unsigned FULL = 0xffffffffu, SENT = 0xffffffffu;
    const int z = blockIdx.y;
    const int b = dir_only >= 0 ? z : (z >> 1);
    const int dir = dir_only >= 0 ? dir_only : (z & 1);
    // NQ / NT: this pair's lengths; the layout of the sorted clouds and boxes is that of the padded sizes
    const int NQ = pair_len(dir == 0 ? len_x : len_y, b, dir == 0 ? P1 : P2);
    const int NT = pair_len(dir == 0 ? len_y : len_x, b, dir == 0 ? P2 : P1);
    const int lane = threadIdx.x & 31;
    const int base = (blockIdx.x * PR_QUERY_WARPS + (threadIdx.x >> 5)) * 32 * R;  // first sorted position of the warp
    if (base >= NQ || NT == 0) return;  // whole warp (no target: chamfer_finalize_kernel writes the zero result)
    const int P1p = soa_padded(P1), P2p = soa_padded(P2);
    const int NQp = dir == 0 ? P1p : P2p;
    const float *__restrict__ QS = dir == 0 ? soa_x + (size_t)b * 4 * P1p : soa_y + (size_t)b * 4 * P2p;
    const float *__restrict__ TS = dir == 0 ? soa_y + (size_t)b * 4 * P2p : soa_x + (size_t)b * 4 * P1p;
    const PrBox *__restrict__ b0 = dir == 0 ? box_y + (size_t)b * pr_boxes(P2) : box_x + (size_t)b * pr_boxes(P1);
    const int NTc = dir == 0 ? P2 : P1;
    const int nb0 = pr_nb0(NTc), nb1 = pr_nb1(NTc), nb2 = pr_nb2(NTc);
    const PrBox *__restrict__ b1 = b0 + nb0, *__restrict__ b2 = b1 + nb1;
    u64 *__restrict__ keys = dir == 0 ? keys_x + (size_t)b * P1 : keys_y + (size_t)b * P2;
    int *__restrict__ list = dir == 0 ? rescue_x + (size_t)b * P1 : rescue_y + (size_t)b * P2;
    const float INF = __int_as_float(0x7f800000);

    bool valid[R];  // positions NQ .. padded end hold +inf padding (inert); beyond the padded end: clamped, inert
    float qx[R], qy[R], qz[R], best[R];
    int qorig[R], barg[R];  // (best, barg): smallest distance so far and the lowest ORIGINAL index that attains it
#pragma unroll
    for (int r = 0; r < R; ++r) {
        const int p = base + r * 32 + lane;
        valid[r] = p < NQ;
        const int pc = min(p, NQp - 1);
        const float *qp = QS + (size_t)(pc >> 4) * 64 + (pc & 15);
        qx[r] = qp[0], qy[r] = qp[16], qz[r] = qp[32];
        qorig[r] = __float_as_int(qp[48]);
        best[r] = valid[r] ? INF : -INF;
        barg[r] = 0x7fffffff;
    }
    bool rescue = (bad_flags[2 * b] | bad_flags[2 * b + 1]) != 0;  // non-finite input: everything takes the exact scan
    if (!rescue) {
        // the warp's query box
        unsigned olx = SENT, oly = SENT, olz = SENT, ohx = 0u, ohy = 0u, ohz = 0u;
#pragma unroll
        for (int r = 0; r < R; ++r)
            if (valid[r]) {
                olx = min(olx, pr_ord(qx[r])), oly = min(oly, pr_ord(qy[r])), olz = min(olz, pr_ord(qz[r]));
                ohx = max(ohx, pr_ord(qx[r])), ohy = max(ohy, pr_ord(qy[r])), ohz = max(ohz, pr_ord(qz[r]));
            }
        const float wlx = pr_unord(__reduce_min_sync(FULL, olx)), wly = pr_unord(__reduce_min_sync(FULL, oly));
        const float wlz = pr_unord(__reduce_min_sync(FULL, olz)), whx = pr_unord(__reduce_max_sync(FULL, ohx));
        const float why = pr_unord(__reduce_max_sync(FULL, ohy)), whz = pr_unord(__reduce_max_sync(FULL, ohz));
        u64 qx2[R], qy2[R], qz2[R];
#pragma unroll
        for (int r = 0; r < R; ++r) qx2[r] = pack2(qx[r], qx[r]), qy2[r] = pack2(qy[r], qy[r]), qz2[r] = pack2(qz[r], qz[r]);
        unsigned wbest = 0x7f800000u;  // bit pattern of the largest `best` among the warp's live queries
        int scans = 0;
        const int scan_cap = max(64, pr_nb0(NT) >> 3);
        bool bail = false;

        int st1 = 0, st2 = 0, st3 = 0, stA = 0, stB = 0, stL = 0;
        (void)st1, (void)st2, (void)st3, (void)stA, (void)stB, (void)stL;
        unsigned k2 = SENT;
        if (lane < nb2) k2 = __float_as_uint(pr_lb(b2[lane].lo, b2[lane].hi, wlx, wly, wlz, whx, why, whz));
        while (!bail) {
            const unsigned m2 = __reduce_min_sync(FULL, k2);
            if (m2 > wbest) break;
            const int n2 = __ffs(__ballot_sync(FULL, k2 == m2)) - 1;
            if (lane == n2) k2 = SENT;
            ++st1;
            const int c1 = n2 * PR_FAN + lane;
            unsigned k1 = SENT;
            if (c1 < nb1) k1 = __float_as_uint(pr_lb(b1[c1].lo, b1[c1].hi, wlx, wly, wlz, whx, why, whz));
            while (!bail) {
                const unsigned m1 = __reduce_min_sync(FULL, k1);
                if (m1 > wbest) break;
                const int n1 = __ffs(__ballot_sync(FULL, k1 == m1)) - 1;
                if (lane == n1) k1 = SENT;
                ++st2;
                const int node1 = n2 * PR_FAN + n1;
                const int c0 = node1 * PR_FAN + lane;
                unsigned k0 = SENT;
                if (c0 < nb0) k0 = __float_as_uint(pr_lb(b0[c0].lo, b0[c0].hi, wlx, wly, wlz, whx, why, whz));
                while (true) {
                    const unsigned m0 = __reduce_min_sync(FULL, k0);
                    if (m0 > wbest) break;
                    const int l0 = __ffs(__ballot_sync(FULL, k0 == m0)) - 1;
                    if (lane == l0) k0 = SENT;
                    ++st3;
                    const int c = node1 * PR_FAN + l0;
                    const float4 blo = b0[c].lo, bhi = b0[c].hi;
                    bool want = false;
#pragma unroll
                    for (int r = 0; r < R; ++r)
                        want |= pr_lb(blo, bhi, qx[r], qy[r], qz[r], qx[r], qy[r], qz[r]) <= best[r];
#ifdef PTK_PR_STATS
                    {
                        const unsigned wb = __ballot_sync(FULL, want);
                        if (wb & 0xffffu) ++stA;
                        if (wb >> 16) ++stB;
                        stL += __popc(wb);
                    }
#endif
                    if (!__any_sync(FULL, want)) continue;
                    if (++scans > scan_cap) {
                        bail = true;
                        break;
                    }
                    // scan the leaf: 16 targets, uniform addresses, the defining arithmetic on packed pairs
                    const float *__restrict__ cp = TS + (size_t)c * 64;
                    float m[R], d[R][PR_CHUNK];
#pragma unroll
                    for (int r = 0; r < R; ++r) m[r] = INF;
#pragma unroll
                    for (int g = 0; g < PR_CHUNK / 4; ++g) {
                        const ulonglong2 tx = *reinterpret_cast<const ulonglong2 *>(cp + g * 4);
                        const ulonglong2 ty = *reinterpret_cast<const ulonglong2 *>(cp + 16 + g * 4);
                        const ulonglong2 tz = *reinterpret_cast<const ulonglong2 *>(cp + 32 + g * 4);
#pragma unroll
                        for (int r = 0; r < R; ++r) {
                            const u64 dxa = sub2(qx2[r], tx.x), dxb = sub2(qx2[r], tx.y);
                            const u64 dya = sub2(qy2[r], ty.x), dyb = sub2(qy2[r], ty.y);
                            const u64 dza = sub2(qz2[r], tz.x), dzb = sub2(qz2[r], tz.y);
                            u64 da = mul2(dxa, dxa), db = mul2(dxb, dxb);
                            da = fma2(dya, dya, da);
                            db = fma2(dyb, dyb, db);
                            da = fma2(dza, dza, da);
                            db = fma2(dzb, dzb, db);
                            unpack2(da, d[r][4 * g], d[r][4 * g + 1]);
                            unpack2(db, d[r][4 * g + 2], d[r][4 * g + 3]);
                            m[r] = min3f(m[r], d[r][4 * g], d[r][4 * g + 1]);
                            m[r] = min3f(m[r], d[r][4 * g + 2], d[r][4 * g + 3]);
                        }
                    }
                    bool touch = false;
#pragma unroll
                    for (int r = 0; r < R; ++r) touch |= m[r] <= best[r];
                    if (__any_sync(FULL, touch)) {
                        // some query improves or ties: lowest original index among this leaf's exact minima
                        int a[R];
#pragma unroll
                        for (int r = 0; r < R; ++r) a[r] = 0x7fffffff;
#pragma unroll
                        for (int g = 0; g < PR_CHUNK / 4; ++g) {
                            const int4 id = *reinterpret_cast<const int4 *>(cp + 48 + g * 4);
#pragma unroll
                            for (int r = 0; r < R; ++r) {
                                a[r] = d[r][4 * g] == m[r] ? min(a[r], id.x) : a[r];
                                a[r] = d[r][4 * g + 1] == m[r] ? min(a[r], id.y) : a[r];
                                a[r] = d[r][4 * g + 2] == m[r] ? min(a[r], id.z) : a[r];
                                a[r] = d[r][4 * g + 3] == m[r] ? min(a[r], id.w) : a[r];
                            }
                        }
#pragma unroll
                        for (int r = 0; r < R; ++r)
                            if (m[r] < best[r] || (m[r] == best[r] && a[r] < barg[r])) {
                                best[r] = m[r];
                                barg[r] = a[r];
                            }
                    }
                    unsigned mine = 0u;
#pragma unroll
                    for (int r = 0; r < R; ++r) mine = max(mine, valid[r] ? __float_as_uint(best[r]) : 0u);
                    wbest = __reduce_max_sync(FULL, mine);
                }
            }
        }
        if (bail) rescue = true;
        PR_STAT(0, 1);
        PR_STAT(1, st1);
        PR_STAT(2, st2);
        PR_STAT(3, st3);
        PR_STAT(4, scans);
        PR_STAT(5, bail ? 1 : 0);
        PR_STAT(6, max(stA, stB));  // leaf scans if each 16-query half walked its own leaves
        PR_STAT(7, stL);            // (lane, leaf) pairs that wanted the scan
    }
#pragma unroll
    for (int r = 0; r < R; ++r) {
        if (!valid[r]) continue;
        if (rescue || !(best[r] < INF)) {
            keys[qorig[r]] = ~0ull;  // the rescue scan merges with a 64-bit atomicMin
            const unsigned int pos = atomicAdd(&rescue_count[2 * b + dir], 1u);
            list[pos] = qorig[r];
        } else {
            keys[qorig[r]] = ((u64)__float_as_uint(best[r]) << 32) | (unsigned int)barg[r];
        }
    }
}

}  // namespace ptk
