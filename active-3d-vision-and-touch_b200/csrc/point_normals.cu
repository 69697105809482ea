// Point-cloud normals and local coordinate frames for sm_100a: PyTorch3D 0.5.0's estimate_pointcloud_normals and
// estimate_pointcloud_local_coord_frames, on the idx / dist of ptk_knn_fwd_lengths(points, points, lengths, lengths,
// K), and their gradient into the points.  Contract in include/ptk.h (ptk_point_frames_fwd), design and cost in
// DESIGN.md K1e.
//
// One thread per query i of cloud b, K' = min(K, l) neighbours q_k = p[idx[b,i,k]]:
//     d_k = q_k - p_i,  m = (1/K') sum d_k,  e_k = d_k - m,  C = (1/K') sum e_k e_k^T
// (two passes relative to the query: C is translation invariant, and d_k is small where q_k and p_i are close), a
// cyclic Jacobi eigensolver with PN_SWEEPS sweeps in registers, then the sign rule over a third pass.  pn_frame states
// that arithmetic once for the forward and both backward forms, with every product and sum pinned (no contraction
// left to the compiler), so the backward recomputes the forward's eigensystem bit for bit and the deterministic
// backward's two passes see the same terms.
#include "det_accum.cuh"
#include "nn_common.cuh"

namespace ptk {

constexpr int PN_THREADS = 128;
constexpr int PN_SWEEPS = 6;  // 18 rotations: the off-diagonal of a 3x3 is at rounding level after 4 in practice

__device__ __forceinline__ float pn_dot(const float a[3], const float b[3]) {
    return __fmaf_rn(a[2], b[2], __fmaf_rn(a[1], b[1], __fmul_rn(a[0], b[0])));
}

// a x b
__device__ __forceinline__ void pn_cross(const float a[3], const float b[3], float c[3]) {
    c[0] = __fmaf_rn(a[1], b[2], -__fmul_rn(a[2], b[1]));
    c[1] = __fmaf_rn(a[2], b[0], -__fmul_rn(a[0], b[2]));
    c[2] = __fmaf_rn(a[0], b[1], -__fmul_rn(a[1], b[0]));
}

__device__ __forceinline__ void pn_normalise(float v[3]) {
    const float r = __fsqrt_rn(pn_dot(v, v));
#pragma unroll
    for (int d = 0; d < 3; ++d) v[d] = __fdiv_rn(v[d], r);
}

// d_k = q_k - p_i of slot k
__device__ __forceinline__ int pn_rel(const float *__restrict__ pb, const int32_t *__restrict__ ir, const float p[3],
                                      int k, float d[3]) {
    const int j = ir[k];
#pragma unroll
    for (int c = 0; c < 3; ++c) d[c] = __fsub_rn(pb[(size_t)j * 3 + c], p[c]);
    return j;
}

// One Jacobi rotation of the symmetric a (both triangles stored) in the (P, Q) plane, accumulated into the columns of
// v (Numerical Recipes' jacobi: t = sgn(theta) / (|theta| + sqrt(theta^2 + 1)), theta = (a_qq - a_pp) / (2 a_pq)).
// An overflowing theta gives t = 0: the rotation only clears a_pq, which is below rounding of the diagonal gap.
template <int P, int Q>
__device__ __forceinline__ void pn_rotate(float (&a)[3][3], float (&v)[3][3]) {
    constexpr int R = 3 - P - Q;
    const float apq = a[P][Q];
    if (apq == 0.0f) return;
    const float theta = __fdiv_rn(__fsub_rn(a[Q][Q], a[P][P]), __fmul_rn(2.0f, apq));
    const float t = __fdiv_rn(copysignf(1.0f, theta), __fadd_rn(fabsf(theta), __fsqrt_rn(__fmaf_rn(theta, theta, 1.0f))));
    const float c = __fdiv_rn(1.0f, __fsqrt_rn(__fmaf_rn(t, t, 1.0f)));
    const float s = __fmul_rn(t, c);
    const float tapq = __fmul_rn(t, apq);
    a[P][P] = __fsub_rn(a[P][P], tapq);
    a[Q][Q] = __fadd_rn(a[Q][Q], tapq);
    a[P][Q] = a[Q][P] = 0.0f;
    const float arp = a[R][P], arq = a[R][Q];
    a[R][P] = a[P][R] = __fmaf_rn(c, arp, -__fmul_rn(s, arq));
    a[R][Q] = a[Q][R] = __fmaf_rn(s, arp, __fmul_rn(c, arq));
#pragma unroll
    for (int k = 0; k < 3; ++k) {
        const float vp = v[k][P], vq = v[k][Q];
        v[k][P] = __fmaf_rn(c, vp, -__fmul_rn(s, vq));
        v[k][Q] = __fmaf_rn(s, vp, __fmul_rn(c, vq));
    }
}

// eigenpairs P and Q into ascending order (a stable compare-exchange: equal eigenvalues keep their order)
template <int P, int Q>
__device__ __forceinline__ void pn_order(float (&lam)[3], float (&v)[3][3]) {
    if (lam[P] > lam[Q]) {
        const float t = lam[P];
        lam[P] = lam[Q];
        lam[Q] = t;
#pragma unroll
        for (int k = 0; k < 3; ++k) {
            const float u = v[k][P];
            v[k][P] = v[k][Q];
            v[k][Q] = u;
        }
    }
}

// The eigensystem of query i: lam ascending, v0 / v1 / v2 the unit eigenvectors with the solver's signs (v0
// normalised, v2 orthogonalised against it and normalised, v1 = v2 x v0), s0 / s2 the sign-rule factors (+1 without
// disambiguation), p the query and m the neighbour mean relative to it.  false when a slot k < K' has a non-finite
// K-NN distance (the query's outputs are NaN).
struct PnFrame {
    float lam[3], v0[3], v1[3], v2[3], p[3], m[3];
    float s0, s2;
};

__device__ __forceinline__ bool pn_frame(const float *__restrict__ pb, const int32_t *__restrict__ ir,
                                         const float *__restrict__ dr, int i, int Kp, bool disambiguate, PnFrame &f) {
    bool ok = true;
    float sum[3] = {0.0f, 0.0f, 0.0f}, d[3];
#pragma unroll
    for (int c = 0; c < 3; ++c) f.p[c] = pb[(size_t)i * 3 + c];
    for (int k = 0; k < Kp; ++k) {
        ok &= isfinite(dr[k]);
        pn_rel(pb, ir, f.p, k, d);
#pragma unroll
        for (int c = 0; c < 3; ++c) sum[c] = __fadd_rn(sum[c], d[c]);
    }
    if (!ok) return false;
    const float kp = (float)Kp;
#pragma unroll
    for (int c = 0; c < 3; ++c) f.m[c] = __fdiv_rn(sum[c], kp);
    float a[3][3] = {{0.0f, 0.0f, 0.0f}, {0.0f, 0.0f, 0.0f}, {0.0f, 0.0f, 0.0f}};
    for (int k = 0; k < Kp; ++k) {
        pn_rel(pb, ir, f.p, k, d);
        float e[3];
#pragma unroll
        for (int c = 0; c < 3; ++c) e[c] = __fsub_rn(d[c], f.m[c]);
#pragma unroll
        for (int r = 0; r < 3; ++r)
#pragma unroll
            for (int c = r; c < 3; ++c) a[r][c] = __fmaf_rn(e[r], e[c], a[r][c]);
    }
#pragma unroll
    for (int r = 0; r < 3; ++r)
#pragma unroll
        for (int c = r; c < 3; ++c) a[c][r] = a[r][c] = __fdiv_rn(a[r][c], kp);

    float v[3][3] = {{1.0f, 0.0f, 0.0f}, {0.0f, 1.0f, 0.0f}, {0.0f, 0.0f, 1.0f}};
#pragma unroll
    for (int sweep = 0; sweep < PN_SWEEPS; ++sweep) {
        pn_rotate<0, 1>(a, v);
        pn_rotate<0, 2>(a, v);
        pn_rotate<1, 2>(a, v);
    }
    float lam[3] = {a[0][0], a[1][1], a[2][2]};
    pn_order<0, 1>(lam, v);
    pn_order<1, 2>(lam, v);
    pn_order<0, 1>(lam, v);
#pragma unroll
    for (int c = 0; c < 3; ++c) {
        f.lam[c] = lam[c];
        f.v0[c] = v[c][0];
        f.v2[c] = v[c][2];
    }
    pn_normalise(f.v0);
    const float w = pn_dot(f.v2, f.v0);
#pragma unroll
    for (int c = 0; c < 3; ++c) f.v2[c] = __fmaf_rn(-w, f.v0[c], f.v2[c]);
    pn_normalise(f.v2);
    pn_cross(f.v2, f.v0, f.v1);

    f.s0 = f.s2 = 1.0f;
    if (disambiguate) {
        int n0 = 0, n2 = 0;
        for (int k = 0; k < Kp; ++k) {
            pn_rel(pb, ir, f.p, k, d);
            n0 += pn_dot(f.v0, d) > 0.0f;
            n2 += pn_dot(f.v2, d) > 0.0f;
        }
        f.s0 = 2 * n0 < Kp ? -1.0f : 1.0f;
        f.s2 = 2 * n2 < Kp ? -1.0f : 1.0f;
    }
    return true;
}

// The output frame (n, y, z): with the sign rule n = s0 v0, z = s2 v2, y = n x z; without it (v0, v1, v2)
__device__ __forceinline__ void pn_axes(const PnFrame &f, bool disambiguate, float n[3], float y[3], float z[3]) {
#pragma unroll
    for (int c = 0; c < 3; ++c) {
        n[c] = f.s0 * f.v0[c];
        z[c] = f.s2 * f.v2[c];
    }
    if (disambiguate) {
        pn_cross(n, z, y);
    } else {
#pragma unroll
        for (int c = 0; c < 3; ++c) y[c] = f.v1[c];
    }
}

// grid = (ceil(P / PN_THREADS), B).  normals (B,P,3) and / or curvatures (B,P,3) with frames (B,P,3,3), columns
// (n, y, z): frames[b,i,r,c] is component r of axis c.
__global__ void __launch_bounds__(PN_THREADS)
point_frames_fwd_kernel(const float *__restrict__ points, const int64_t *__restrict__ lengths,
                        const int32_t *__restrict__ idx, const float *__restrict__ dist, int P, int K, int disambiguate,
                        float *__restrict__ normals, float *__restrict__ curvatures, float *__restrict__ frames) {
    pdl_wait();
    const int b = blockIdx.y;
    const int i = blockIdx.x * PN_THREADS + threadIdx.x;
    if (i >= P) return;
    const int L = pair_len(lengths, b, P);
    const size_t o = (size_t)b * P + i;
    float n[3], y[3], z[3], lam[3];
    PnFrame f;
    if (i >= L) {  // padded query: zeros
#pragma unroll
        for (int c = 0; c < 3; ++c) n[c] = y[c] = z[c] = lam[c] = 0.0f;
    } else if (!pn_frame(points + (size_t)b * P * 3, idx + o * K, dist + o * K, i, min(K, L), disambiguate != 0, f)) {
        const float nan = __int_as_float(0x7fffffff);
#pragma unroll
        for (int c = 0; c < 3; ++c) n[c] = y[c] = z[c] = lam[c] = nan;
    } else {
        pn_axes(f, disambiguate != 0, n, y, z);
#pragma unroll
        for (int c = 0; c < 3; ++c) lam[c] = f.lam[c];
    }
    if (normals)
#pragma unroll
        for (int c = 0; c < 3; ++c) normals[o * 3 + c] = n[c];
    if (frames) {
#pragma unroll
        for (int c = 0; c < 3; ++c) {
            curvatures[o * 3 + c] = lam[c];
            frames[o * 9 + c * 3 + 0] = n[c];
            frames[o * 9 + c * 3 + 1] = y[c];
            frames[o * 9 + c * 3 + 2] = z[c];
        }
    }
}

// ---------------------------------------------------------------------------------------- backward
// The gradient w.r.t. C of query i, symmetrised and divided by K': S = (G + G^T) / K' with G = V (diag(gL) + F o
// (V^T gV)) V^T, F_mn = 1 / (lam_n - lam_m) off the diagonal (linalg.eigh's backward), taken as 0 where lam_n == lam_m
// in fp32 (a repeated eigenspace has no defined gradient; 0 also keeps a zero upstream gradient exactly zero).  gV
// folds the upstream gradients: frames' y = n x z passes z x g_y to n and g_y x n to z, the sign rule passes s0 g_n to
// v0 and s2 g_z to v2; normals add to n.  Any upstream pointer may be NULL (zero).
__device__ __forceinline__ void pn_grad_matrix(const PnFrame &f, bool disambiguate, int Kp,
                                               const float *__restrict__ grad_normals,
                                               const float *__restrict__ grad_curvatures,
                                               const float *__restrict__ grad_frames, size_t o, float S[3][3]) {
    float gv[3][3], gl[3];  // gv[m]: the gradient of eigenvector m
#pragma unroll
    for (int c = 0; c < 3; ++c) {
#pragma unroll
        for (int m = 0; m < 3; ++m) gv[m][c] = grad_frames ? grad_frames[o * 9 + c * 3 + m] : 0.0f;
        if (grad_normals) gv[0][c] = __fadd_rn(gv[0][c], grad_normals[o * 3 + c]);
        gl[c] = grad_curvatures ? grad_curvatures[o * 3 + c] : 0.0f;
    }
    if (disambiguate) {
        float n[3], y[3], z[3], t0[3], t2[3];
        pn_axes(f, true, n, y, z);
        pn_cross(z, gv[1], t0);
        pn_cross(gv[1], n, t2);
#pragma unroll
        for (int c = 0; c < 3; ++c) {
            gv[0][c] = f.s0 * __fadd_rn(gv[0][c], t0[c]);
            gv[2][c] = f.s2 * __fadd_rn(gv[2][c], t2[c]);
            gv[1][c] = 0.0f;
        }
    }
    const float *vm[3] = {f.v0, f.v1, f.v2};
    float M[3][3];
#pragma unroll
    for (int m = 0; m < 3; ++m)
#pragma unroll
        for (int n = 0; n < 3; ++n) {
            if (m == n) {
                M[m][n] = gl[m];
            } else {
                const float gap = __fsub_rn(f.lam[n], f.lam[m]);
                M[m][n] = gap != 0.0f ? __fdiv_rn(pn_dot(vm[m], gv[n]), gap) : 0.0f;
            }
        }
    // T = V (M + M^T), S = T V^T / K'
    float T[3][3];
#pragma unroll
    for (int a = 0; a < 3; ++a)
#pragma unroll
        for (int n = 0; n < 3; ++n) {
            float acc = 0.0f;
#pragma unroll
            for (int m = 0; m < 3; ++m) acc = __fmaf_rn(vm[m][a], __fadd_rn(M[m][n], M[n][m]), acc);
            T[a][n] = acc;
        }
    const float kp = (float)Kp;
#pragma unroll
    for (int a = 0; a < 3; ++a)
#pragma unroll
        for (int b = 0; b < 3; ++b) {
            float acc = 0.0f;
#pragma unroll
            for (int n = 0; n < 3; ++n) acc = __fmaf_rn(T[a][n], vm[n][b], acc);
            S[a][b] = __fdiv_rn(acc, kp);
        }
}

// The term of slot k, S (q_k - mean), for neighbour j (returned)
__device__ __forceinline__ int pn_term(const PnFrame &f, const float S[3][3], const float *__restrict__ pb,
                                       const int32_t *__restrict__ ir, int k, float t[3]) {
    float d[3], e[3];
    const int j = pn_rel(pb, ir, f.p, k, d);
#pragma unroll
    for (int c = 0; c < 3; ++c) e[c] = __fsub_rn(d[c], f.m[c]);
#pragma unroll
    for (int r = 0; r < 3; ++r) t[r] = pn_dot(S[r], e);
    return j;
}

// Query i's eigensystem and S; false for a query that passes no gradient (padded, or NaN outputs)
__device__ __forceinline__ bool pn_query_grad(const float *__restrict__ points, const int64_t *__restrict__ lengths,
                                              const int32_t *__restrict__ idx, const float *__restrict__ dist, int b,
                                              int i, int P, int K, int disambiguate,
                                              const float *__restrict__ grad_normals,
                                              const float *__restrict__ grad_curvatures,
                                              const float *__restrict__ grad_frames, int &Kp, PnFrame &f,
                                              float S[3][3]) {
    const int L = pair_len(lengths, b, P);
    if (i >= L) return false;
    const size_t o = (size_t)b * P + i;
    Kp = min(K, L);
    if (!pn_frame(points + (size_t)b * P * 3, idx + o * K, dist + o * K, i, Kp, disambiguate != 0, f)) return false;
    pn_grad_matrix(f, disambiguate != 0, Kp, grad_normals, grad_curvatures, grad_frames, o, S);
    return true;
}

// Default backward, grid = (ceil(P / PN_THREADS), B): one thread per query, each slot's term added to its neighbour's
// row with fp32 atomics (grad_points zeroed by the caller)
__global__ void __launch_bounds__(PN_THREADS)
point_frames_bwd_kernel(const float *__restrict__ points, const int64_t *__restrict__ lengths,
                        const int32_t *__restrict__ idx, const float *__restrict__ dist, int P, int K, int disambiguate,
                        const float *__restrict__ grad_normals, const float *__restrict__ grad_curvatures,
                        const float *__restrict__ grad_frames, float *__restrict__ grad_points) {
    pdl_wait();
    const int b = blockIdx.y;
    const int i = blockIdx.x * PN_THREADS + threadIdx.x;
    if (i >= P) return;
    int Kp;
    PnFrame f;
    float S[3][3], t[3];
    if (!pn_query_grad(points, lengths, idx, dist, b, i, P, K, disambiguate, grad_normals, grad_curvatures, grad_frames,
                       Kp, f, S))
        return;
    const float *pb = points + (size_t)b * P * 3;
    const int32_t *ir = idx + ((size_t)b * P + i) * K;
    float *gb = grad_points + (size_t)b * P * 3;
    for (int k = 0; k < Kp; ++k) {
        const int j = pn_term(f, S, pb, ir, k, t);
#pragma unroll
        for (int c = 0; c < 3; ++c) atomicAdd(gb + (size_t)j * 3 + c, t[c]);
    }
}

// Deterministic form (det_accum.cuh): M_b over the finite terms of cloud b, n = l + 1 (a query's K' neighbours are
// distinct, so a row receives at most l terms).
// phase 1, grid = (ceil(P / PN_THREADS), B): M_b (atomicMax into mbits[b], zeroed by the caller), accumulators and
// grad_points rows zeroed
__global__ void __launch_bounds__(PN_THREADS)
point_frames_bwd_det_max_kernel(const float *__restrict__ points, const int64_t *__restrict__ lengths,
                                const int32_t *__restrict__ idx, const float *__restrict__ dist, int P, int K,
                                int disambiguate, const float *__restrict__ grad_normals,
                                const float *__restrict__ grad_curvatures, const float *__restrict__ grad_frames,
                                float *__restrict__ grad_points, unsigned long long *__restrict__ acc,
                                unsigned int *__restrict__ mbits) {
    pdl_wait();
    const int b = blockIdx.y;
    const int i = blockIdx.x * PN_THREADS + threadIdx.x;
    float m = 0.0f;
    if (i < P) {
        det_zero_row(acc, grad_points, (size_t)b * P + i);
        int Kp;
        PnFrame f;
        float S[3][3], t[3];
        if (pn_query_grad(points, lengths, idx, dist, b, i, P, K, disambiguate, grad_normals, grad_curvatures,
                          grad_frames, Kp, f, S)) {
            const float *pb = points + (size_t)b * P * 3;
            const int32_t *ir = idx + ((size_t)b * P + i) * K;
            for (int k = 0; k < Kp; ++k) {
                pn_term(f, S, pb, ir, k, t);
                m = fmaxf(m, fmaxf(det_abs_finite(t[0]), fmaxf(det_abs_finite(t[1]), det_abs_finite(t[2]))));
            }
        }
    }
    det_block_max<PN_THREADS>(m, mbits + b);
}

// phase 2, grid = (ceil(P / PN_THREADS), B): quantise and add into the neighbour's row (non-finite terms into
// grad_points)
__global__ void __launch_bounds__(PN_THREADS)
point_frames_bwd_det_add_kernel(const float *__restrict__ points, const int64_t *__restrict__ lengths,
                                const int32_t *__restrict__ idx, const float *__restrict__ dist, int P, int K,
                                int disambiguate, const float *__restrict__ grad_normals,
                                const float *__restrict__ grad_curvatures, const float *__restrict__ grad_frames,
                                float *__restrict__ grad_points, unsigned long long *__restrict__ acc,
                                const unsigned int *__restrict__ mbits, DetBound nb) {
    pdl_wait();
    const int b = blockIdx.y;
    const int i = blockIdx.x * PN_THREADS + threadIdx.x;
    if (i >= P) return;
    int Kp;
    PnFrame f;
    float S[3][3], t[3];
    if (!pn_query_grad(points, lengths, idx, dist, b, i, P, K, disambiguate, grad_normals, grad_curvatures, grad_frames,
                       Kp, f, S))
        return;
    const double scale = det_scale(mbits, nb, b);
    const float *pb = points + (size_t)b * P * 3;
    const int32_t *ir = idx + ((size_t)b * P + i) * K;
    for (int k = 0; k < Kp; ++k) {
        const size_t r = ((size_t)b * P + pn_term(f, S, pb, ir, k, t)) * 3;
#pragma unroll
        for (int c = 0; c < 3; ++c) det_add(acc + r + c, grad_points + r + c, t[c], scale);
    }
}

// ---------------------------------------------------------------------------------------- host side
static int pn_check(const float *points, const int32_t *idx, const float *dist, int64_t B, int64_t P, int64_t K,
                    const char *what) {
    PTK_REQUIRE(points && idx && dist, PTK_ERR_SHAPE, "%s: null points / idx / dist pointer", what);
    PTK_REQUIRE(B > 0 && P > 0 && B <= 65535 && P < (1LL << 31) / 9, PTK_ERR_SHAPE, "%s: bad sizes (B=%lld, P=%lld)",
                what, (long long)B, (long long)P);
    PTK_REQUIRE(K >= 1 && K <= PTK_KNN_MAX_K, PTK_ERR_SHAPE, "%s: K=%lld outside [1, %d]", what, (long long)K,
                PTK_KNN_MAX_K);
    PTK_REQUIRE(P * K < (1LL << 31), PTK_ERR_SHAPE, "%s: P * K too large for 32-bit indexing", what);
    return PTK_OK;
}

static dim3 pn_grid(int64_t B, int64_t P) { return dim3((unsigned)ceil_div(P, PN_THREADS), (unsigned)B); }

}  // namespace ptk

using namespace ptk;

extern "C" int ptk_point_frames_fwd(const float *points, const int64_t *lengths, const int32_t *idx, const float *dist,
                                    int64_t B, int64_t P, int64_t K, int disambiguate, float *normals,
                                    float *curvatures, float *frames, ptk_stream_t stream) {
    PTK_NVTX("ptk_point_frames_fwd");
    int rc = pn_check(points, idx, dist, B, P, K, "point_frames_fwd");
    if (rc) return rc;
    PTK_REQUIRE((normals || frames) && !curvatures == !frames, PTK_ERR_SHAPE,
                "point_frames_fwd: null output pointer (normals, or curvatures and frames)");
    launch_pdl(point_frames_fwd_kernel, pn_grid(B, P), dim3(PN_THREADS), 0, as_stream(stream), points, lengths, idx,
               dist, (int)P, (int)K, disambiguate, normals, curvatures, frames);
    PTK_CHECK_LAUNCH();
    return PTK_OK;
}

extern "C" int ptk_point_frames_bwd(const float *points, const int64_t *lengths, const int32_t *idx, const float *dist,
                                    int64_t B, int64_t P, int64_t K, int disambiguate, const float *grad_normals,
                                    const float *grad_curvatures, const float *grad_frames, float *grad_points,
                                    ptk_stream_t stream) {
    PTK_NVTX("ptk_point_frames_bwd");
    int rc = pn_check(points, idx, dist, B, P, K, "point_frames_bwd");
    if (rc) return rc;
    PTK_REQUIRE(grad_points, PTK_ERR_SHAPE, "point_frames_bwd: null grad_points pointer");
    cudaStream_t st = as_stream(stream);
    PTK_CHECK_CUDA(cudaMemsetAsync(grad_points, 0, sizeof(float) * (size_t)B * P * 3, st));
    if (!grad_normals && !grad_curvatures && !grad_frames) return PTK_OK;
    launch_pdl(point_frames_bwd_kernel, pn_grid(B, P), dim3(PN_THREADS), 0, st, points, lengths, idx, dist, (int)P,
               (int)K, disambiguate, grad_normals, grad_curvatures, grad_frames, grad_points);
    PTK_CHECK_LAUNCH();
    return PTK_OK;
}

extern "C" int ptk_point_frames_bwd_det(const float *points, const int64_t *lengths, const int32_t *idx,
                                        const float *dist, int64_t B, int64_t P, int64_t K, int disambiguate,
                                        const float *grad_normals, const float *grad_curvatures,
                                        const float *grad_frames, float *grad_points, void *workspace,
                                        size_t workspace_bytes, ptk_stream_t stream) {
    PTK_NVTX("ptk_point_frames_bwd_det");
    int rc = pn_check(points, idx, dist, B, P, K, "point_frames_bwd_det");
    if (rc) return rc;
    PTK_REQUIRE(grad_points, PTK_ERR_SHAPE, "point_frames_bwd_det: null grad_points pointer");
    rc = det_check_workspace(workspace, workspace_bytes, ptk_knn1_bwd_det_workspace_bytes(B, P, P),
                             "point_frames_bwd_det");
    if (rc) return rc;
    cudaStream_t st = as_stream(stream);
    if (!grad_normals && !grad_curvatures && !grad_frames) {
        PTK_CHECK_CUDA(cudaMemsetAsync(grad_points, 0, sizeof(float) * (size_t)B * P * 3, st));
        return PTK_OK;
    }
    DetWs w;
    PTK_CHECK_CUDA(det_begin(workspace, B, P, st, w));
    const DetBound nb = det_bound_len(lengths, P);
    launch_pdl(point_frames_bwd_det_max_kernel, pn_grid(B, P), dim3(PN_THREADS), 0, st, points, lengths, idx, dist,
               (int)P, (int)K, disambiguate, grad_normals, grad_curvatures, grad_frames, grad_points, w.acc_a, w.mbits);
    PTK_CHECK_LAUNCH();
    launch_pdl(point_frames_bwd_det_add_kernel, pn_grid(B, P), dim3(PN_THREADS), 0, st, points, lengths, idx, dist,
               (int)P, (int)K, disambiguate, grad_normals, grad_curvatures, grad_frames, grad_points, w.acc_a,
               (const unsigned int *)w.mbits, nb);
    PTK_CHECK_LAUNCH();
    det_launch_convert<PN_THREADS>(w, nb, B, grad_points, P, nullptr, 0, st);
    PTK_CHECK_LAUNCH();
    return PTK_OK;
}
