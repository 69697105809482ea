// Chamfer nearest-neighbour kernels, second generation (shared by chamfer.cu and tools/chamfer_tune.cu).
//
//   chamfer_nn_filter_kernel   3-FFMA "expansion" FILTER + exact recheck (the fast path)
//   chamfer_nn_exact2_kernel   the defining 6-op arithmetic with packed FP32x2 instructions
//
// Both return, per query, EXACTLY the (distance, index) the defining arithmetic of chamfer_kernel.cuh
// (sqdist(): fma(dz,dz, fma(dy,dy, dx*dx)), strict '<' in ascending target order) returns.
//
// Filter idea.  min_t |q-t|^2 = |q|^2 + min_t ( |t|^2 - 2 q.t ).  The bracket costs 3 FFMA per
// (query, target) instead of 6 FP32-pipe instructions, but it cancels: its rounding error is
// O(u R^2) (R = cloud radius), not O(u d^2).  It is therefore used only to find WHERE the minimum
// can be:
//   * clouds are translated to the centre c of their joint bounding box (shrinks R; the exact
//     arithmetic keeps using the untranslated coordinates);
//   * per query the scan keeps the smallest chunk minimum `best` (chunk = CHUNK consecutive targets, 64 in
//     the library's TMA scan), the chunk that produced it, and the smallest chunk minimum of any OTHER chunk, `second`;
//   * afterwards the recorded chunk is re-evaluated with the exact arithmetic (first minimum wins);
//   * if second > best + thr no target outside that chunk can beat or tie it (thr bounds every
//     rounding error involved, see PairAux below), so the result is final.  Otherwise the
//     query is "ambiguous" (near-tie or exact tie across chunks): it is appended to a per-cloud
//     rescue list and chamfer_nn_exact2_kernel re-scans the whole target range for it with the
//     exact arithmetic (64-bit atomicMin merge).  Correctness never depends on the filter:
//     thr = +inf (non-finite or extreme input) sends every query down the exact path.
#pragma once
#include "chamfer_kernel.cuh"

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

// Per cloud pair: centre c of the joint bounding box and the ambiguity threshold of the filter.
//
// Notation: u = 2^-24; qc = fl(q - c), tc = fl(t - c) the translated points (what the filter sees);
// M^2 >= |pc|^2 for every translated point of both clouds; a(t) the computed filter value;
// D = |q-t|^2 in exact arithmetic, d_def the defining arithmetic's result, bd = d_def of the exact
// arg-min e* inside the recorded chunk, b* the target that gave `best`.
//   (E1) filter:       |a(t) - (|tc|^2 - 2 qc.tc)| <= 12 u M^2   (3 roundings in tt, 3 in the FMA chain, every
//                      partial sum is bounded by |tc|^2 + 2|qc||tc| <= 3 M^2)
//   (E2) translation:  | |qc-tc|^2 - D | <= 4 u M sqrt(D) + 4 u^2 M^2      (each point moves by <= u M)
//   (E3) definition:   |d_def - D| <= 5.01 u D                             (2 roundings in each difference, 3 after)
// Claim: a(t) - a(b*) > thr_q  =>  d_def(t) > bd.  Proof sketch: assume d_def(t) <= bd <= d_def(b*).  By (E3)
// D_t <= bd (1+5.01u) and D_b* >= bd (1-5u); by (E1) and a(b*) <= a(e*), D_b* <= bd + 25 u M^2.  Chaining
// (E1), (E2) for t and b*:  a(t) - a(b*) <= 24 u M^2 + 10.01 u bd + 4 u M (sqrt(D_t) + sqrt(D_b*)) + 8 u^2 M^2
//                                         <= 25.1 u M^2 + 26.1 u bd          (2 M sqrt(bd) <= M^2/4 + 4 bd).
// The kernels use thr_q = 32 u M^2 + 32 u bd: the spare 7 u M^2 covers the rounding of `best + thr_q` itself
// (|best| <= 4 M^2) and second-order terms.  aux.thr = 32 u M^2 = 2^-19 M^2, rounded up.
// The chunk width does not enter: the claim compares single targets t and b*, e* is the exact arg-min of whatever
// range is rechecked, and `second` is a minimum over single targets outside it.  A wider chunk only moves near-ties
// inside the rechecked range, where the exact arithmetic settles them.
// Non-finite input, M^2 > 1e30 or M^2 < 1e-30 (squares would overflow / lose relative accuracy to underflow)
// set thr = +inf: every query then takes the exact path.
struct PairAux {
    float cx, cy, cz, thr;
};
constexpr float FILTER_THR_BD = 1.9073486e-6f;  // 32 u = 2^-19

// Ragged batches: the points of cloud b that exist, len[b] clamped to [0, P] (P when the caller passed no lengths).
// Row strides stay those of the padded (B, P, 3) tensor; only the counts of queries and targets become per pair, so
// padding points are never read into a result, a bound or the filter's certificate.
__device__ __forceinline__ int pair_len(const int64_t *__restrict__ len, int b, int P) {
    if (len == nullptr) return P;
    const long long v = len[b];
    return v < 0 ? 0 : (v > P ? P : (int)v);
}

__global__ void __launch_bounds__(1024)
chamfer_bounds_kernel(const float *__restrict__ x, const float *__restrict__ y, int P1, int P2,
                      const int64_t *__restrict__ len_x, const int64_t *__restrict__ len_y,
                      PairAux *__restrict__ aux, unsigned int *__restrict__ rescue_count) {
    pdl_wait();  // launched with programmatic stream serialization (ptk_common.cuh)
    const int b = blockIdx.x;
    const int tid = threadIdx.x;
    const int L1 = pair_len(len_x, b, P1), L2 = pair_len(len_y, b, P2);
    const float PINF = __int_as_float(0x7f800000), NINF = __int_as_float(0xff800000);
    __shared__ float sred[7][32];
    __shared__ float sctr[3];
    __shared__ int sbad;
    if (tid == 0) sbad = 0;

    // pass 1: bounding box of both clouds.  Thread t handles elements t, t+1024, ...; its coordinate
    // index (e % 3) advances by 1024 % 3 == 1 per step.
    float lo[3] = {PINF, PINF, PINF}, hi[3] = {NINF, NINF, NINF};
    bool bad = false;
    for (int s = 0; s < 2; ++s) {
        const float *p = s == 0 ? x + (size_t)b * P1 * 3 : y + (size_t)b * P2 * 3;
        const int n = (s == 0 ? L1 : L2) * 3;
        // eight loads in flight per thread: at small batches this single CTA per pair is latency-bound
        for (int e0 = tid; e0 < n; e0 += 8 * 1024) {
            float v[8];
#pragma unroll
            for (int u = 0; u < 8; ++u) v[u] = e0 + u * 1024 < n ? p[e0 + u * 1024] : p[tid % 3];
#pragma unroll
            for (int u = 0; u < 8; ++u) {
                const int e = e0 + u * 1024 < n ? e0 + u * 1024 : tid % 3;  // the filler repeats a real element
                const int c = e % 3;
                bad |= !(fabsf(v[u]) <= 3.0e38f);  // NaN or Inf
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
        sctr[tid] = l <= h ? 0.5f * l + 0.5f * h : 0.f;  // no finite point (both clouds empty): not NaN
    }
    __syncthreads();
    const float cx = sctr[0], cy = sctr[1], cz = sctr[2];

    // pass 2: M^2 = max |fl(p - c)|^2 over both clouds, every operation rounded up
    float m2 = 0.f;
    for (int s = 0; s < 2; ++s) {
        const float *p = s == 0 ? x + (size_t)b * P1 * 3 : y + (size_t)b * P2 * 3;
        const int n = s == 0 ? L1 : L2;
#pragma unroll 4
        for (int i = tid; i < n; i += 1024) {
            const float dx = __fsub_rn(p[i * 3 + 0], cx), dy = __fsub_rn(p[i * 3 + 1], cy), dz = __fsub_rn(p[i * 3 + 2], cz);
            m2 = fmaxf(m2, __fmaf_ru(dz, dz, __fmaf_ru(dy, dy, __fmul_ru(dx, dx))));
        }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) m2 = fmaxf(m2, __shfl_xor_sync(0xffffffffu, m2, o));
    if ((tid & 31) == 0) sred[6][tid >> 5] = m2;
    __syncthreads();
    if (tid == 0) {
        for (int w = 1; w < 32; ++w) m2 = fmaxf(m2, sred[6][w]);
        PairAux a;
        a.cx = cx;
        a.cy = cy;
        a.cz = cz;
        a.thr = __fmul_ru(m2, FILTER_THR_BD);
        if (sbad || !(m2 <= 1.0e30f) || !(m2 >= 1.0e-30f)) {
            a.cx = a.cy = a.cz = 0.f;
            a.thr = PINF;  // every query takes the exact path
        }
        aux[b] = a;
        if (rescue_count) rescue_count[2 * b] = rescue_count[2 * b + 1] = 0u;
    }
}

// R queries per thread, CHUNK targets per lazy-argmin chunk, THREADS per CTA, MINB resident CTAs/SM.
// Shared tile: TT targets as SoA x[], y[], z[], tt[] (translated coordinates, tt = |t|^2).
template <int R, int CHUNK, int THREADS, int MINB, int TT, bool PACKED>
__global__ void __launch_bounds__(THREADS, MINB)
chamfer_nn_filter_kernel(const float *__restrict__ x, const float *__restrict__ y, int P1, int P2,
                         int split_len, int n_split, const PairAux *__restrict__ aux,
                         u64 *__restrict__ keys_x, u64 *__restrict__ keys_y, int dir_only,
                         int *__restrict__ rescue_x, int *__restrict__ rescue_y,
                         unsigned int *__restrict__ rescue_count, unsigned int *__restrict__ rescue_flag_x,
                         unsigned int *__restrict__ rescue_flag_y) {
    static_assert(CHUNK % 16 == 0 && TT % CHUNK == 0, "tile must hold whole chunks of 16-target bodies");
    const int z = blockIdx.z;
    const int b = dir_only >= 0 ? z : (z >> 1);
    const int dir = dir_only >= 0 ? dir_only : (z & 1);
    const int NQ = dir == 0 ? P1 : P2;
    const int NT = dir == 0 ? P2 : P1;
    const float *__restrict__ Q = dir == 0 ? x + (size_t)b * P1 * 3 : y + (size_t)b * P2 * 3;
    const float *__restrict__ T = dir == 0 ? y + (size_t)b * P2 * 3 : x + (size_t)b * P1 * 3;
    u64 *__restrict__ keys = dir == 0 ? keys_x + (size_t)b * P1 : keys_y + (size_t)b * P2;

    const int q0 = blockIdx.x * (THREADS * R);
    if (q0 >= NQ) return;
    const int t_begin = blockIdx.y * split_len;
    if (t_begin >= NT) return;
    const int t_end = min(NT, t_begin + split_len);
    const int tid = threadIdx.x;
    const PairAux ax = aux[b];
    const float INF = __int_as_float(0x7f800000);

    __shared__ __align__(16) float sx[TT];
    __shared__ __align__(16) float sy[TT];
    __shared__ __align__(16) float sz[TT];
    __shared__ __align__(16) float st[TT];

    float mqx[R], mqy[R], mqz[R];  // -2 (q - c)
    float best[R], sec[R];
    int bchunk[R];
#pragma unroll
    for (int r = 0; r < R; ++r) {
        const int qi = min(q0 + r * THREADS + tid, NQ - 1);
        const float ax_ = -2.0f * __fsub_rn(Q[(size_t)qi * 3 + 0], ax.cx);
        const float ay_ = -2.0f * __fsub_rn(Q[(size_t)qi * 3 + 1], ax.cy);
        const float az_ = -2.0f * __fsub_rn(Q[(size_t)qi * 3 + 2], ax.cz);
        mqx[r] = ax_;
        mqy[r] = ay_;
        mqz[r] = az_;
        best[r] = INF;
        sec[r] = INF;
        bchunk[r] = t_begin / CHUNK;
    }

    for (int tile = t_begin; tile < t_end; tile += TT) {
        const int n = min(TT, t_end - tile);
        const int npad = ((n + CHUNK - 1) / CHUNK) * CHUNK;
        __syncthreads();
        const float *__restrict__ src = T + (size_t)tile * 3;
        for (int p = tid; p < npad; p += THREADS) {
            float tx = 0.f, ty = 0.f, tz = 0.f, tt = INF;  // padding never wins
            if (p < n) {
                tx = __fsub_rn(src[p * 3 + 0], ax.cx);
                ty = __fsub_rn(src[p * 3 + 1], ax.cy);
                tz = __fsub_rn(src[p * 3 + 2], ax.cz);
                tt = __fmaf_rn(tz, tz, __fmaf_rn(ty, ty, __fmul_rn(tx, tx)));
            }
            sx[p] = tx;
            sy[p] = ty;
            sz[p] = tz;
            st[p] = tt;
        }
        __syncthreads();
        const int nchunks = npad / CHUNK;
        const int chunk0 = tile / CHUNK;
        for (int c = 0; c < nchunks; ++c) {
            float m[R];
#pragma unroll
            for (int r = 0; r < R; ++r) m[r] = INF;
#pragma unroll 1
            for (int sub = 0; sub < CHUNK / 16; ++sub) {
#pragma unroll
            for (int g4 = 0; g4 < 4; ++g4) {
                const int g = sub * 4 + g4;
                if (PACKED) {
                    const ulonglong2 tx = *reinterpret_cast<const ulonglong2 *>(&sx[c * CHUNK + g * 4]);
                    const ulonglong2 ty = *reinterpret_cast<const ulonglong2 *>(&sy[c * CHUNK + g * 4]);
                    const ulonglong2 tz = *reinterpret_cast<const ulonglong2 *>(&sz[c * CHUNK + g * 4]);
                    const ulonglong2 tt = *reinterpret_cast<const ulonglong2 *>(&st[c * CHUNK + g * 4]);
#pragma unroll
                    for (int r = 0; r < R; ++r) {
                        const u64 qx2 = pack2(mqx[r], mqx[r]), qy2 = pack2(mqy[r], mqy[r]), qz2 = pack2(mqz[r], mqz[r]);
                        u64 a = fma2(qx2, tx.x, tt.x);
                        u64 c2 = fma2(qx2, tx.y, tt.y);
                        a = fma2(qy2, ty.x, a);
                        c2 = fma2(qy2, ty.y, c2);
                        a = fma2(qz2, tz.x, a);
                        c2 = fma2(qz2, tz.y, c2);
                        float a0, a1, a2, a3;
                        unpack2(a, a0, a1);
                        unpack2(c2, a2, a3);
                        m[r] = min3f(m[r], a0, a1);
                        m[r] = min3f(m[r], a2, a3);
                    }
                } else {
                    const float4 tx = *reinterpret_cast<const float4 *>(&sx[c * CHUNK + g * 4]);
                    const float4 ty = *reinterpret_cast<const float4 *>(&sy[c * CHUNK + g * 4]);
                    const float4 tz = *reinterpret_cast<const float4 *>(&sz[c * CHUNK + g * 4]);
                    const float4 tt = *reinterpret_cast<const float4 *>(&st[c * CHUNK + g * 4]);
#pragma unroll
                    for (int r = 0; r < R; ++r) {
                        const float a0 = __fmaf_rn(mqz[r], tz.x, __fmaf_rn(mqy[r], ty.x, __fmaf_rn(mqx[r], tx.x, tt.x)));
                        const float a1 = __fmaf_rn(mqz[r], tz.y, __fmaf_rn(mqy[r], ty.y, __fmaf_rn(mqx[r], tx.y, tt.y)));
                        const float a2 = __fmaf_rn(mqz[r], tz.z, __fmaf_rn(mqy[r], ty.z, __fmaf_rn(mqx[r], tx.z, tt.z)));
                        const float a3 = __fmaf_rn(mqz[r], tz.w, __fmaf_rn(mqy[r], ty.w, __fmaf_rn(mqx[r], tx.w, tt.w)));
                        m[r] = min3f(m[r], a0, a1);
                        m[r] = min3f(m[r], a2, a3);
                    }
                }
            }
            }
#pragma unroll
            for (int r = 0; r < R; ++r) {
                sec[r] = fminf(sec[r], fmaxf(m[r], best[r]));
                bchunk[r] = m[r] < best[r] ? chunk0 + c : bchunk[r];
                best[r] = fminf(best[r], m[r]);
            }
        }
    }

    // Exact recheck of the recorded chunk -> tentative key (always a true candidate).  Ambiguous
    // queries are additionally queued for chamfer_nn_exact2_kernel (list mode).
    int *__restrict__ rescue = dir == 0 ? rescue_x + (size_t)b * P1 : rescue_y + (size_t)b * P2;
    unsigned int *__restrict__ rflag = dir == 0 ? rescue_flag_x + (size_t)b * P1 : rescue_flag_y + (size_t)b * P2;
#pragma unroll
    for (int r = 0; r < R; ++r) {
        const int qi = q0 + r * THREADS + tid;
        if (qi >= NQ) continue;
        const float qx = Q[(size_t)qi * 3 + 0], qy = Q[(size_t)qi * 3 + 1], qz = Q[(size_t)qi * 3 + 2];
        const int j0 = bchunk[r] * CHUNK;
        const int j1 = min(j0 + CHUNK, t_end);
        float bd = INF;
        int arg = j0;
        for (int j = j0; j < j1; ++j) {
            const float d = sqdist(qx, qy, qz, T[(size_t)j * 3], T[(size_t)j * 3 + 1], T[(size_t)j * 3 + 2]);
            if (d < bd) {
                bd = d;
                arg = j;
            }
        }
        const u64 key = ((u64)__float_as_uint(bd) << 32) | (unsigned int)arg;
        if (n_split > 1)
            atomicMin(&keys[qi], key);
        else
            keys[qi] = key;
        if (!(sec[r] > best[r] + __fmaf_ru(bd, FILTER_THR_BD, ax.thr))) {
            // with a split target range several CTAs may flag the same query: queue it once
            if (n_split == 1 || atomicExch(&rflag[qi], 1u) == 0u)
                rescue[atomicAdd(&rescue_count[2 * b + dir], 1u)] = qi;
        }
    }
}

// ------------------------------------------------------------------------------------------------
// TMA-staged variant of the filter scan.
//
// chamfer_prep_kernel writes, once per forward, every cloud as four padded SoA arrays
// [X | Y | Z | TT] of translated coordinates (TT = |t|^2, padding: 0,0,0,+inf).  The scan then streams
// target tiles straight into shared memory with cp.async.bulk (TMA, mbarrier complete_tx), double
// buffered: no staging arithmetic and no load latency inside the scan, one CTA barrier per tile that only
// waits for warp skew.
constexpr int SOA_PAD = 64;  // clouds are padded to a multiple of this many points

__host__ __device__ inline int soa_padded(int P) { return (P + SOA_PAD - 1) / SOA_PAD * SOA_PAD; }

// grid (ceil(Ppad_max / 256), 2 * B): blockIdx.y = 2 * b + cloud
__global__ void __launch_bounds__(256)
chamfer_prep_kernel(const float *__restrict__ x, const float *__restrict__ y, int P1, int P2,
                    const int64_t *__restrict__ len_x, const int64_t *__restrict__ len_y,
                    const PairAux *__restrict__ aux, float *__restrict__ soa_x, float *__restrict__ soa_y,
                    u64 *__restrict__ keys_x, u64 *__restrict__ keys_y, unsigned int *__restrict__ flag_x,
                    unsigned int *__restrict__ flag_y, int init_keys) {
    pdl_wait();  // launched with programmatic stream serialization (ptk_common.cuh)
    const int b = blockIdx.y >> 1, cloud = blockIdx.y & 1;
    const int P = cloud == 0 ? P1 : P2;
    const int Pp = soa_padded(P);
    const int i = blockIdx.x * 256 + threadIdx.x;
    if (i >= Pp) return;
    const float *src = (cloud == 0 ? x + (size_t)b * P1 * 3 : y + (size_t)b * P2 * 3);
    float *dst = (cloud == 0 ? soa_x + (size_t)b * 4 * Pp : soa_y + (size_t)b * 4 * Pp);
    const PairAux ax = aux[b];
    // points past the cloud's length are padding like those past P: the scan's tiles round up to whole chunks and
    // read up to a chunk past the length
    float tx = 0.f, ty = 0.f, tz = 0.f, tt = __int_as_float(0x7f800000);
    if (i < pair_len(cloud == 0 ? len_x : len_y, b, P)) {
        tx = __fsub_rn(src[i * 3 + 0], ax.cx);
        ty = __fsub_rn(src[i * 3 + 1], ax.cy);
        tz = __fsub_rn(src[i * 3 + 2], ax.cz);
        tt = __fmaf_rn(tz, tz, __fmaf_rn(ty, ty, __fmul_rn(tx, tx)));
    }
    dst[i] = tx;
    dst[Pp + i] = ty;
    dst[2 * Pp + i] = tz;
    dst[3 * Pp + i] = tt;
    // split target ranges merge by atomicMin on the key and dedup their rescue entries through the flag: this
    // point's slots start at "nothing found" / "not queued" (three memsets per forward before)
    if (init_keys && i < P) {
        u64 *keys = cloud == 0 ? keys_x : keys_y;
        unsigned int *flag = cloud == 0 ? flag_x : flag_y;
        if (keys) keys[(size_t)b * P + i] = ~0ull;
        if (flag) flag[(size_t)b * P + i] = 0u;
    }
}

__device__ __forceinline__ uint32_t smem_addr(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_wait_parity(uint32_t bar, uint32_t parity) {
    uint32_t done;
    do {
        asm volatile(
            "{\n\t"
            ".reg .pred p;\n\t"
            "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
            "selp.u32 %0, 1, 0, p;\n\t"
            "}" : "=r"(done) : "r"(bar), "r"(parity) : "memory");
    } while (!done);
}

template <int R, int CHUNK, int THREADS, int MINB, int TT>
__global__ void __launch_bounds__(THREADS, MINB)
chamfer_nn_filter_tma_kernel(const float *__restrict__ x, const float *__restrict__ y, int P1, int P2,
                             const int64_t *__restrict__ len_x, const int64_t *__restrict__ len_y,
                             int split_len, int n_split, const PairAux *__restrict__ aux,
                             const float *__restrict__ soa_x, const float *__restrict__ soa_y,
                             u64 *__restrict__ keys_x, u64 *__restrict__ keys_y, int dir_only,
                             int *__restrict__ rescue_x, int *__restrict__ rescue_y,
                             unsigned int *__restrict__ rescue_count, unsigned int *__restrict__ rescue_flag_x,
                             unsigned int *__restrict__ rescue_flag_y) {
    pdl_wait();  // launched with programmatic stream serialization (ptk_common.cuh)
    static_assert((CHUNK == 16 || CHUNK == 32 || CHUNK == 64) && TT % CHUNK == 0 && SOA_PAD % CHUNK == 0, "tile must hold whole chunks");
    const int z = blockIdx.z;
    const int b = dir_only >= 0 ? z : (z >> 1);
    const int dir = dir_only >= 0 ? dir_only : (z & 1);
    // NQ / NT: this pair's lengths (the SoA and AoS strides below keep using P1 / P2).  The exits below come before any
    // query load, so NQ >= 1 and NT >= 1 past them; a chunk that straddles NT fails `j1 - j0 == CHUNK` in the recheck.
    const int NQ = pair_len(dir == 0 ? len_x : len_y, b, dir == 0 ? P1 : P2);
    const int NT = pair_len(dir == 0 ? len_y : len_x, b, dir == 0 ? P2 : P1);
    const int P1p = soa_padded(P1), P2p = soa_padded(P2);
    const int NQp = dir == 0 ? P1p : P2p, NTp = dir == 0 ? P2p : P1p;
    const float *__restrict__ Q = dir == 0 ? x + (size_t)b * P1 * 3 : y + (size_t)b * P2 * 3;
    const float *__restrict__ T = dir == 0 ? y + (size_t)b * P2 * 3 : x + (size_t)b * P1 * 3;
    const float *__restrict__ QS = dir == 0 ? soa_x + (size_t)b * 4 * P1p : soa_y + (size_t)b * 4 * P2p;
    const float *__restrict__ TS = dir == 0 ? soa_y + (size_t)b * 4 * P2p : soa_x + (size_t)b * 4 * P1p;
    u64 *__restrict__ keys = dir == 0 ? keys_x + (size_t)b * P1 : keys_y + (size_t)b * P2;

    const int q0 = blockIdx.x * (THREADS * R);
    if (q0 >= NQ) return;
    const int t_begin = blockIdx.y * split_len;
    if (t_begin >= NT) return;
    const int t_end = min(NT, t_begin + split_len);
    const int tid = threadIdx.x;
    const PairAux ax = aux[b];
    const float INF = __int_as_float(0x7f800000);

    __shared__ __align__(128) float sbuf[2][4][TT];
    __shared__ __align__(8) u64 mbar[2];
    const uint32_t bar0 = smem_addr(&mbar[0]), bar1 = smem_addr(&mbar[1]);
    const int ntiles = (t_end - t_begin + TT - 1) / TT;
    auto issue = [&](int it) {  // one thread: request tile `it` into buffer it & 1
        const int tile = t_begin + it * TT;
        const int n = min(TT, t_end - tile);
        const uint32_t bytes = (uint32_t)((n + CHUNK - 1) / CHUNK * CHUNK) * 4u;
        const uint32_t bar = (it & 1) ? bar1 : bar0;
        asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(4u * bytes) : "memory");
#pragma unroll
        for (int a = 0; a < 4; ++a)
            asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                         ::"r"(smem_addr(&sbuf[it & 1][a][0])), "l"(TS + (size_t)a * NTp + tile), "r"(bytes), "r"(bar)
                         : "memory");
    };
    if (tid == 0) {
        asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(bar0));
        asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(bar1));
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        issue(0);
        if (ntiles > 1) issue(1);
    }

    float mqx[R], mqy[R], mqz[R];  // -2 (q - c)
    float best[R], sec[R];
    int bchunk[R];
#pragma unroll
    for (int r = 0; r < R; ++r) {
        const int qi = min(q0 + r * THREADS + tid, NQ - 1);
        mqx[r] = -2.0f * QS[qi];
        mqy[r] = -2.0f * QS[NQp + qi];
        mqz[r] = -2.0f * QS[2 * NQp + qi];
        best[r] = INF;
        sec[r] = INF;
        bchunk[r] = t_begin / CHUNK;
    }
    __syncthreads();  // barrier initialisation visible to every waiter

    for (int it = 0; it < ntiles; ++it) {
        const int tile = t_begin + it * TT;
        const int n = min(TT, t_end - tile);
        const int nchunks = (n + CHUNK - 1) / CHUNK;
        const int chunk0 = tile / CHUNK;
        mbar_wait_parity((it & 1) ? bar1 : bar0, (uint32_t)((it >> 1) & 1));
        const float *sx = sbuf[it & 1][0], *sy = sbuf[it & 1][1], *sz = sbuf[it & 1][2], *st = sbuf[it & 1][3];
        // One fully unrolled body per chunk: the chunk minimum starts from the chunk's first values (no +inf operand,
        // no reset), and the bookkeeping is straight-line code the scheduler can slot between the FFMA2s of the other
        // queries.  Per query and 64 targets: 96 FFMA2, 31 FMNMX3 + 1 FMNMX for the minimum, 5 bookkeeping instructions.
        for (int c = 0; c < nchunks; ++c) {
            float m[R];
#pragma unroll
            for (int g4 = 0; g4 < CHUNK / 4; ++g4) {
                const int o = c * CHUNK + g4 * 4;
                const ulonglong2 tx = *reinterpret_cast<const ulonglong2 *>(&sx[o]);
                const ulonglong2 ty = *reinterpret_cast<const ulonglong2 *>(&sy[o]);
                const ulonglong2 tz = *reinterpret_cast<const ulonglong2 *>(&sz[o]);
                const ulonglong2 tt = *reinterpret_cast<const ulonglong2 *>(&st[o]);
#pragma unroll
                for (int r = 0; r < R; ++r) {
                    const u64 qx2 = pack2(mqx[r], mqx[r]), qy2 = pack2(mqy[r], mqy[r]), qz2 = pack2(mqz[r], mqz[r]);
                    u64 a = fma2(qx2, tx.x, tt.x);
                    u64 c2 = fma2(qx2, tx.y, tt.y);
                    a = fma2(qy2, ty.x, a);
                    c2 = fma2(qy2, ty.y, c2);
                    a = fma2(qz2, tz.x, a);
                    c2 = fma2(qz2, tz.y, c2);
                    float a0, a1, a2, a3;
                    unpack2(a, a0, a1);
                    unpack2(c2, a2, a3);
                    if (g4 == 0) {
                        m[r] = fminf(min3f(a0, a1, a2), a3);
                    } else {
                        m[r] = min3f(m[r], a0, a1);
                        m[r] = min3f(m[r], a2, a3);
                    }
                }
            }
            const int cid = chunk0 + c;
#pragma unroll
            for (int r = 0; r < R; ++r) {
                sec[r] = fminf(sec[r], fmaxf(m[r], best[r]));
                bchunk[r] = m[r] < best[r] ? cid : bchunk[r];
                best[r] = fminf(best[r], m[r]);
            }
        }
        __syncthreads();  // every warp is done with this buffer
        if (tid == 0 && it + 2 < ntiles) issue(it + 2);
    }

    // Exact recheck of the recorded chunk.  It needs the untranslated coordinates, so it reads the caller's AoS cloud,
    // not the translated SoA copy.  Each thread reads its own chunk, so every load of a warp touches 32 different
    // cache lines: with 4-byte loads the recheck of 64-target chunks cost more L1 bandwidth than the wider chunks
    // saved.  Whole chunks are therefore read with 256-bit loads (3 per 8 targets) when the cloud is 32-byte aligned,
    // with float4 loads (3 per 4 targets) when it is 16-byte aligned; a chunk then starts on such a boundary because
    // CHUNK * 12 is a multiple of 32.
    static_assert(CHUNK % 8 == 0, "vector recheck reads whole groups of 8 targets");
    const bool t_aligned = (reinterpret_cast<uintptr_t>(T) & 15) == 0;
    const bool t_aligned32 = (reinterpret_cast<uintptr_t>(T) & 31) == 0;
    int *__restrict__ rescue = dir == 0 ? rescue_x + (size_t)b * P1 : rescue_y + (size_t)b * P2;
    unsigned int *__restrict__ rflag = dir == 0 ? rescue_flag_x + (size_t)b * P1 : rescue_flag_y + (size_t)b * P2;
#pragma unroll
    for (int r = 0; r < R; ++r) {
        const int qi = q0 + r * THREADS + tid;
        if (qi >= NQ) continue;
        const float qx = Q[(size_t)qi * 3 + 0], qy = Q[(size_t)qi * 3 + 1], qz = Q[(size_t)qi * 3 + 2];
        const int j0 = bchunk[r] * CHUNK;
        const int j1 = min(j0 + CHUNK, t_end);
        float bd = INF;
        int arg = j0;
        auto consider = [&](float tx, float ty, float tz, int j) {
            const float d = sqdist(qx, qy, qz, tx, ty, tz);
            if (d < bd) {
                bd = d;
                arg = j;
            }
        };
        if (t_aligned32 && j1 - j0 == CHUNK) {
            const float *tp = T + (size_t)j0 * 3;
#pragma unroll 2
            for (int k = 0; k < CHUNK / 8; ++k) {
                float v[24];
#pragma unroll
                for (int h = 0; h < 3; ++h)
                    asm("ld.global.nc.v8.f32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
                        : "=f"(v[8 * h]), "=f"(v[8 * h + 1]), "=f"(v[8 * h + 2]), "=f"(v[8 * h + 3]), "=f"(v[8 * h + 4]),
                          "=f"(v[8 * h + 5]), "=f"(v[8 * h + 6]), "=f"(v[8 * h + 7])
                        : "l"(tp + 24 * k + 8 * h));
#pragma unroll
                for (int i = 0; i < 8; ++i) consider(v[3 * i], v[3 * i + 1], v[3 * i + 2], j0 + 8 * k + i);
            }
        } else if (t_aligned && j1 - j0 == CHUNK) {
            const float4 *__restrict__ t4 = reinterpret_cast<const float4 *>(T + (size_t)j0 * 3);
#pragma unroll 4
            for (int k = 0; k < CHUNK / 4; ++k) {
                const float4 u = __ldg(t4 + 3 * k), v = __ldg(t4 + 3 * k + 1), w = __ldg(t4 + 3 * k + 2);
                consider(u.x, u.y, u.z, j0 + 4 * k);
                consider(u.w, v.x, v.y, j0 + 4 * k + 1);
                consider(v.z, v.w, w.x, j0 + 4 * k + 2);
                consider(w.y, w.z, w.w, j0 + 4 * k + 3);
            }
        } else {
            for (int j = j0; j < j1; ++j) consider(T[(size_t)j * 3], T[(size_t)j * 3 + 1], T[(size_t)j * 3 + 2], j);
        }
        const u64 key = ((u64)__float_as_uint(bd) << 32) | (unsigned int)arg;
        if (n_split > 1)
            atomicMin(&keys[qi], key);
        else
            keys[qi] = key;
        if (!(sec[r] > best[r] + __fmaf_ru(bd, FILTER_THR_BD, ax.thr))) {
            if (n_split == 1 || atomicExch(&rflag[qi], 1u) == 0u)
                rescue[atomicAdd(&rescue_count[2 * b + dir], 1u)] = qi;
        }
    }
}


// The defining arithmetic with packed FP32x2 instructions (two targets per instruction): same
// results as chamfer_nn_kernel bit for bit, half the FP32-pipe issue slots.
//
// Direct mode (rescue_* == nullptr): CTA blockIdx.x owns queries [q0, q0 + THREADS*R).
// List mode: it owns entries [q0, q0 + THREADS*R) of the cloud's rescue list (query ids queued by
// chamfer_nn_filter_kernel), merges with atomicMin, and exits at once when the list is shorter.
// A CTA with at most THREADS entries runs the one-query-per-thread body instead of wasting R-1 slots.
template <int R, int CHUNK, int THREADS>
__device__ __forceinline__ void exact2_body(const float *__restrict__ Q, const float *__restrict__ T, int NT,
                                            int t_begin, int t_end, const int (&qidx)[R], const bool (&valid)[R],
                                            u64 *__restrict__ keys, bool atomic_merge, float *sx, float *sy,
                                            float *sz, int coff = 0, int cstride = 1) {
    // coff/cstride: this thread only scans chunks coff, coff + cstride, ... of every tile (used when
    // several warps share one short query list and split the targets; merged by atomicMin)
    const int tid = threadIdx.x;
    const float INF = __int_as_float(0x7f800000);
    u64 qx[R], qy[R], qz[R];
    float best[R];
    int bchunk[R];
#pragma unroll
    for (int r = 0; r < R; ++r) {
        const int qi = qidx[r];
        const float a = Q[(size_t)qi * 3 + 0], bq = Q[(size_t)qi * 3 + 1], c = Q[(size_t)qi * 3 + 2];
        qx[r] = pack2(a, a);
        qy[r] = pack2(bq, bq);
        qz[r] = pack2(c, c);
        best[r] = INF;
        bchunk[r] = t_begin / CHUNK;
    }

    for (int tile = t_begin; tile < t_end; tile += CH_TT) {
        const int n = min(CH_TT, t_end - tile);
        __syncthreads();
        const int npad = ((n + CHUNK - 1) / CHUNK) * CHUNK;
        const float *__restrict__ src = T + (size_t)tile * 3;
        // eight loads in flight per thread: in list mode only a few CTAs are resident and this staging is
        // latency-bound (ncu: 255 us rescue pass, long-scoreboard stalls) unless the loads are batched
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
        __syncthreads();
        const int nchunks = npad / CHUNK;
        const int chunk0 = tile / CHUNK;
        for (int c = coff; c < nchunks; c += cstride) {
            float m[R];
#pragma unroll
            for (int r = 0; r < R; ++r) m[r] = INF;
#pragma unroll
            for (int g = 0; g < CHUNK / 4; ++g) {
                const ulonglong2 tx = *reinterpret_cast<const ulonglong2 *>(&sx[c * CHUNK + g * 4]);
                const ulonglong2 ty = *reinterpret_cast<const ulonglong2 *>(&sy[c * CHUNK + g * 4]);
                const ulonglong2 tz = *reinterpret_cast<const ulonglong2 *>(&sz[c * CHUNK + g * 4]);
#pragma unroll
                for (int r = 0; r < R; ++r) {
                    const u64 dxa = sub2(qx[r], tx.x), dxb = sub2(qx[r], tx.y);
                    const u64 dya = sub2(qy[r], ty.x), dyb = sub2(qy[r], ty.y);
                    const u64 dza = sub2(qz[r], tz.x), dzb = sub2(qz[r], tz.y);
                    u64 da = mul2(dxa, dxa), db = mul2(dxb, dxb);
                    da = fma2(dya, dya, da);
                    db = fma2(dyb, dyb, db);
                    da = fma2(dza, dza, da);
                    db = fma2(dzb, dzb, db);
                    float d0, d1, d2, d3;
                    unpack2(da, d0, d1);
                    unpack2(db, d2, d3);
                    m[r] = min3f(m[r], d0, d1);
                    m[r] = min3f(m[r], d2, d3);
                }
            }
#pragma unroll
            for (int r = 0; r < R; ++r) {
                bchunk[r] = m[r] < best[r] ? chunk0 + c : bchunk[r];
                best[r] = fminf(best[r], m[r]);
            }
        }
    }

#pragma unroll
    for (int r = 0; r < R; ++r) {
        if (!valid[r]) continue;
        float a, bq, c, dummy;
        unpack2(qx[r], a, dummy);
        unpack2(qy[r], bq, dummy);
        unpack2(qz[r], c, dummy);
        const int j0 = bchunk[r] * CHUNK;
        const int j1 = min(j0 + CHUNK, NT);
        int arg = j0;
        bool found = false;
        for (int j = j0; j < j1; ++j) {
            float d = sqdist(a, bq, c, T[(size_t)j * 3], T[(size_t)j * 3 + 1], T[(size_t)j * 3 + 2]);
            if (!found && d == best[r]) {
                arg = j;
                found = true;
            }
        }
        u64 key = ((u64)__float_as_uint(best[r]) << 32) | (unsigned int)arg;
        if (atomic_merge)
            atomicMin(&keys[qidx[r]], key);
        else
            keys[qidx[r]] = key;
    }
}

template <int R, int CHUNK, int THREADS, int MINB>
__global__ void __launch_bounds__(THREADS, MINB)
chamfer_nn_exact2_kernel(const float *__restrict__ x, const float *__restrict__ y, int P1, int P2,
                         const int64_t *__restrict__ len_x, const int64_t *__restrict__ len_y,
                         int split_len, int n_split, u64 *__restrict__ keys_x,
                         u64 *__restrict__ keys_y, int dir_only, const int *__restrict__ rescue_x,
                         const int *__restrict__ rescue_y, const unsigned int *__restrict__ rescue_count) {
    pdl_wait();  // launched with programmatic stream serialization (ptk_common.cuh)
    const int z = blockIdx.z;
    const int b = dir_only >= 0 ? z : (z >> 1);
    const int dir = dir_only >= 0 ? dir_only : (z & 1);
    const int NQ = pair_len(dir == 0 ? len_x : len_y, b, dir == 0 ? P1 : P2);  // this pair's lengths, as in the filter
    const int NT = pair_len(dir == 0 ? len_y : len_x, b, dir == 0 ? P2 : P1);
    const float *__restrict__ Q = dir == 0 ? x + (size_t)b * P1 * 3 : y + (size_t)b * P2 * 3;
    const float *__restrict__ T = dir == 0 ? y + (size_t)b * P2 * 3 : x + (size_t)b * P1 * 3;
    u64 *__restrict__ keys = dir == 0 ? keys_x + (size_t)b * P1 : keys_y + (size_t)b * P2;

    const bool list_mode = rescue_count != nullptr;
    const int *__restrict__ list = nullptr;
    int NL = NQ;  // number of work items of this cloud/direction
    if (list_mode) {
        list = dir == 0 ? rescue_x + (size_t)b * P1 : rescue_y + (size_t)b * P2;
        NL = (int)min(rescue_count[2 * b + dir], (unsigned int)NQ);
    }
    const int q0 = blockIdx.x * (THREADS * R);
    if (q0 >= NL) return;
    const int t_begin = blockIdx.y * split_len;
    if (t_begin >= NT) return;
    const int t_end = min(NT, t_begin + split_len);
    const int tid = threadIdx.x;
    const bool atomic_merge = list_mode || n_split > 1;

    __shared__ __align__(16) float sx[CH_TT];
    __shared__ __align__(16) float sy[CH_TT];
    __shared__ __align__(16) float sz[CH_TT];

    if (list_mode && NL - q0 <= THREADS) {
        int qidx[1];
        bool valid[1];
        if (NL - q0 <= 32) {
            // at most one warp of queries: every warp takes all of them and 1/nwarps of the chunks
            const int e = q0 + (tid & 31);
            valid[0] = e < NL;
            qidx[0] = list[min(e, NL - 1)];
            exact2_body<1, CHUNK, THREADS>(Q, T, NT, t_begin, t_end, qidx, valid, keys, true, sx, sy, sz, tid >> 5,
                                           THREADS / 32);
            return;
        }
        const int e = q0 + tid;
        valid[0] = e < NL;
        qidx[0] = list[min(e, NL - 1)];
        exact2_body<1, CHUNK, THREADS>(Q, T, NT, t_begin, t_end, qidx, valid, keys, true, sx, sy, sz);
        return;
    }
    int qidx[R];
    bool valid[R];
#pragma unroll
    for (int r = 0; r < R; ++r) {
        const int e = q0 + r * THREADS + tid;
        valid[r] = e < NL;
        const int ec = min(e, NL - 1);
        qidx[r] = list_mode ? list[ec] : ec;
    }
    exact2_body<R, CHUNK, THREADS>(Q, T, NT, t_begin, t_end, qidx, valid, keys, atomic_merge, sx, sy, sz);
}

}  // namespace ptk
