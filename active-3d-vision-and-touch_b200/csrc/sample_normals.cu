// Normals of points sampled from meshes for sm_100a: the return_normals branch of PyTorch3D 0.5.0's
// sample_points_from_meshes, on the face_idx of ptk_sample_fwd, and its gradient into the mesh vertices.  Contract in
// include/ptk.h (ptk_sample_normals_fwd), design and cost in DESIGN.md K3b.
//
// For sample s on face f with corners v0, v1, v2:
//     e1 = v1 - v0, e2 = v2 - v1, c = e1 x e2, r = |c|, q = max(r, eps), n = c / q     (eps = sys.float_info.epsilon)
// Every product, difference and sum is rounded on its own (no FMA contraction), as in sampler.cu's face_area_rn.  The
// backward adds, per sample and corner, the sampler's point term w_k * g_pts and the normal term of the chain
// g_n -> g_c -> (g_e1, g_e2) -> (g_v0, g_v1, g_v2), both computed by sn_terms below so that the default and the
// deterministic forms add the same fp32 values.  This file is separate from sampler.cu so that the sampler's SASS
// stays as it is.
#include "det_accum.cuh"

namespace ptk {

constexpr int SN_THREADS = 256;
constexpr float SN_EPS = 2.220446049250313e-16f;  // sys.float_info.epsilon (2^-52), exact in fp32
constexpr int SN_SMEM_VERTS = 4096;               // default backward: 4096 * 3 floats = 48 KB of shared accumulators
constexpr int SND_SMEM_VERTS = 2048;              // deterministic backward: 2048 * 3 int64 = 48 KB
constexpr int SN_PER_CTA = 2048;                  // backward: samples per CTA (each CTA clears and flushes the mesh)

__device__ __forceinline__ float sn_dot_rn(const float a[3], const float b[3]) {
    return __fadd_rn(__fadd_rn(__fmul_rn(a[0], b[0]), __fmul_rn(a[1], b[1])), __fmul_rn(a[2], b[2]));
}

// a x b, each product and difference rounded on its own
__device__ __forceinline__ void sn_cross_rn(const float a[3], const float b[3], float c[3]) {
    c[0] = __fsub_rn(__fmul_rn(a[1], b[2]), __fmul_rn(a[2], b[1]));
    c[1] = __fsub_rn(__fmul_rn(a[2], b[0]), __fmul_rn(a[0], b[2]));
    c[2] = __fsub_rn(__fmul_rn(a[0], b[1]), __fmul_rn(a[1], b[0]));
}

// the face of sample o (an out-of-range id is clamped, as sample_points_kernel clamps a given one) and its corners
__device__ __forceinline__ void sn_face(const float *__restrict__ vb, const int32_t *__restrict__ faces,
                                        const int32_t *__restrict__ face_idx, int F, size_t o, int vi[3], float v[3][3]) {
    const int f = min(max(face_idx[o], 0), F - 1);
#pragma unroll
    for (int k = 0; k < 3; ++k) {
        vi[k] = faces[f * 3 + k];
#pragma unroll
        for (int d = 0; d < 3; ++d) v[k][d] = vb[(size_t)vi[k] * 3 + d];
    }
}

// e1, e2, c = e1 x e2, the clamped norm q and the unit normal n of corners v; returns r = |c| (NaN stays NaN: the
// comparison r < eps is false, so q = r)
__device__ __forceinline__ float sn_normal(const float v[3][3], float e1[3], float e2[3], float n[3], float &q) {
    float c[3];
#pragma unroll
    for (int d = 0; d < 3; ++d) {
        e1[d] = __fsub_rn(v[1][d], v[0][d]);
        e2[d] = __fsub_rn(v[2][d], v[1][d]);
    }
    sn_cross_rn(e1, e2, c);
    const float r = __fsqrt_rn(sn_dot_rn(c, c));
    q = r < SN_EPS ? SN_EPS : r;
#pragma unroll
    for (int d = 0; d < 3; ++d) n[d] = __fdiv_rn(c[d], q);
    return r;
}

// The per-sample terms of the backward, corner k, component d:
//   pt[k][d] = w_k * g_pts[d]                                (the sampler's term; 0 when g_pts is NULL)
//   nt[k][d] = the normal term: g_c = (g_n - (n . g_n) n) / q when r >= eps (= g_n / r - (c . g_n) c / r^3; at
//              r = eps the clamp passes the gradient through, as clamp_min's backward does), g_c = g_n / eps when
//              r < eps; g_e1 = e2 x g_c, g_e2 = g_c x e1; g_v0 = -g_e1, g_v1 = g_e1 - g_e2, g_v2 = g_e2.
// vi: the corners' vertex ids.
__device__ __forceinline__ void sn_terms(const float *__restrict__ vb, const int32_t *__restrict__ faces,
                                         const int32_t *__restrict__ face_idx, const float *__restrict__ uu,
                                         const float *__restrict__ vv, const float *__restrict__ grad_pts,
                                         const float *__restrict__ grad_n, int F, size_t o, int vi[3], float pt[3][3],
                                         float nt[3][3]) {
    float v[3][3], e1[3], e2[3], n[3], q;
    sn_face(vb, faces, face_idx, F, o, vi, v);
    const float r = sn_normal(v, e1, e2, n, q);
    const float g[3] = {grad_n[o * 3 + 0], grad_n[o * 3 + 1], grad_n[o * 3 + 2]};
    const float s = r >= SN_EPS ? sn_dot_rn(n, g) : 0.0f;
    float gc[3], ge1[3], ge2[3];
#pragma unroll
    for (int d = 0; d < 3; ++d) gc[d] = __fdiv_rn(__fsub_rn(g[d], __fmul_rn(s, n[d])), q);
    sn_cross_rn(e2, gc, ge1);
    sn_cross_rn(gc, e1, ge2);
#pragma unroll
    for (int d = 0; d < 3; ++d) {
        nt[0][d] = -ge1[d];
        nt[1][d] = __fsub_rn(ge1[d], ge2[d]);
        nt[2][d] = ge2[d];
    }
    // barycentric weights: the operations of sample_points_kernel / sample_bwd_kernel
    const float rt = __fsqrt_rn(uu[o]);
    const float vw = vv[o];
    const float w[3] = {__fsub_rn(1.0f, rt), __fmul_rn(rt, __fsub_rn(1.0f, vw)), __fmul_rn(rt, vw)};
#pragma unroll
    for (int k = 0; k < 3; ++k)
#pragma unroll
        for (int d = 0; d < 3; ++d) pt[k][d] = grad_pts ? __fmul_rn(w[k], grad_pts[o * 3 + d]) : 0.0f;
}

// Forward, grid = (ceil(S / SN_THREADS), B): one thread per sample, 12 B out
__global__ void __launch_bounds__(SN_THREADS)
sample_normals_fwd_kernel(const float *__restrict__ verts, int V, const int32_t *__restrict__ faces, int F,
                          const int32_t *__restrict__ face_idx, int S, float *__restrict__ normals) {
    pdl_wait();  // launched with programmatic stream serialization (ptk_common.cuh)
    const int b = blockIdx.y;
    const int s = blockIdx.x * SN_THREADS + threadIdx.x;
    if (s >= S) return;
    const size_t o = (size_t)b * S + s;
    int vi[3];
    float v[3][3], e1[3], e2[3], n[3], q;
    sn_face(verts + (size_t)b * V * 3, faces, face_idx, F, o, vi, v);
    sn_normal(v, e1, e2, n, q);
#pragma unroll
    for (int d = 0; d < 3; ++d) normals[o * 3 + d] = n[d];
}

// Default backward, grid = (ceil(S / SN_PER_CTA), B): both terms of a (sample, corner, component) added, then one
// fp32 atomic; in shared memory while the mesh has at most SN_SMEM_VERTS vertices (then one RED per touched
// component), otherwise straight into grad_verts (zeroed by the caller)
__global__ void __launch_bounds__(SN_THREADS)
sample_normals_bwd_kernel(const float *__restrict__ verts, const int32_t *__restrict__ faces,
                          const int32_t *__restrict__ face_idx, const float *__restrict__ uu,
                          const float *__restrict__ vv, const float *__restrict__ grad_pts,
                          const float *__restrict__ grad_n, int V, int F, int S, float *__restrict__ grad_verts) {
    pdl_wait();
    const int b = blockIdx.y;
    const int tid = threadIdx.x;
    __shared__ float s_acc[SN_SMEM_VERTS * 3];
    const bool in_smem = V <= SN_SMEM_VERTS;
    if (in_smem) {
        for (int k = tid; k < V * 3; k += SN_THREADS) s_acc[k] = 0.0f;
        __syncthreads();
    }
    const float *vb = verts + (size_t)b * V * 3;
    float *gv = grad_verts + (size_t)b * V * 3;
    const int s_begin = blockIdx.x * SN_PER_CTA;
    const int s_end = min(S, s_begin + SN_PER_CTA);
    for (int s = s_begin + tid; s < s_end; s += SN_THREADS) {
        int vi[3];
        float pt[3][3], nt[3][3];
        sn_terms(vb, faces, face_idx, uu, vv, grad_pts, grad_n, F, (size_t)b * S + s, vi, pt, nt);
#pragma unroll
        for (int k = 0; k < 3; ++k)
#pragma unroll
            for (int d = 0; d < 3; ++d) {
                const float c = __fadd_rn(pt[k][d], nt[k][d]);
                if (in_smem)
                    atomicAdd(&s_acc[vi[k] * 3 + d], c);
                else
                    atomicAdd(&gv[(size_t)vi[k] * 3 + d], c);
            }
    }
    if (in_smem) {
        __syncthreads();
        for (int k = tid; k < V * 3; k += SN_THREADS) {
            const float a = s_acc[k];
            if (a != 0.0f) atomicAdd(&gv[k], a);
        }
    }
}

// Deterministic backward (ptk_sample_normals_bwd_det, scheme in det_accum.cuh): every (sample, corner, component) has
// two terms, quantised separately; a vertex receives at most 3 S point terms and 3 S normal terms, so n = 6 S + 1.
// phase 1, grid = (ceil(max(S, V) / SN_THREADS), B): M_b over both kinds (atomicMax into mbits[b], zeroed by the
// caller); accumulators and grad_verts zeroed
__global__ void __launch_bounds__(SN_THREADS)
sample_normals_bwd_det_max_kernel(const float *__restrict__ verts, const int32_t *__restrict__ faces,
                                  const int32_t *__restrict__ face_idx, const float *__restrict__ uu,
                                  const float *__restrict__ vv, const float *__restrict__ grad_pts,
                                  const float *__restrict__ grad_n, int V, int F, int S, float *__restrict__ grad_verts,
                                  unsigned long long *__restrict__ acc, unsigned int *__restrict__ mbits) {
    pdl_wait();
    const int b = blockIdx.y;
    const int i = blockIdx.x * SN_THREADS + threadIdx.x;
    float m = 0.0f;
    if (i < S) {
        int vi[3];
        float pt[3][3], nt[3][3];
        sn_terms(verts + (size_t)b * V * 3, faces, face_idx, uu, vv, grad_pts, grad_n, F, (size_t)b * S + i, vi, pt, nt);
#pragma unroll
        for (int k = 0; k < 3; ++k)
#pragma unroll
            for (int d = 0; d < 3; ++d) m = fmaxf(m, fmaxf(det_abs_finite(pt[k][d]), det_abs_finite(nt[k][d])));
    }
    if (i < V) det_zero_row(acc, grad_verts, (size_t)b * V + i);
    det_block_max<SN_THREADS>(m, mbits + b);
}

// phase 2, grid = (ceil(S / SN_PER_CTA), B): quantise and add both terms.  Meshes of up to SND_SMEM_VERTS vertices are
// accumulated in shared int64 first (exact as well), then one global 64-bit reduction per touched component.
__global__ void __launch_bounds__(SN_THREADS)
sample_normals_bwd_det_add_kernel(const float *__restrict__ verts, const int32_t *__restrict__ faces,
                                  const int32_t *__restrict__ face_idx, const float *__restrict__ uu,
                                  const float *__restrict__ vv, const float *__restrict__ grad_pts,
                                  const float *__restrict__ grad_n, int V, int F, int S, float *__restrict__ grad_verts,
                                  unsigned long long *__restrict__ acc, const unsigned int *__restrict__ mbits,
                                  DetBound nb) {
    pdl_wait();
    const int b = blockIdx.y;
    const int tid = threadIdx.x;
    __shared__ unsigned long long s_acc[SND_SMEM_VERTS * 3];
    const bool in_smem = V <= SND_SMEM_VERTS;
    if (in_smem) {
        for (int k = tid; k < V * 3; k += SN_THREADS) s_acc[k] = 0ull;
        __syncthreads();
    }
    const double scale = det_scale(mbits, nb, b);
    const float *vb = verts + (size_t)b * V * 3;
    float *gv = grad_verts + (size_t)b * V * 3;
    unsigned long long *av = acc + (size_t)b * V * 3;
    const int s_begin = blockIdx.x * SN_PER_CTA;
    const int s_end = min(S, s_begin + SN_PER_CTA);
    for (int s = s_begin + tid; s < s_end; s += SN_THREADS) {
        int vi[3];
        float pt[3][3], nt[3][3];
        sn_terms(vb, faces, face_idx, uu, vv, grad_pts, grad_n, F, (size_t)b * S + s, vi, pt, nt);
#pragma unroll
        for (int k = 0; k < 3; ++k)
#pragma unroll
            for (int d = 0; d < 3; ++d) {
                const size_t e = (size_t)vi[k] * 3 + d;
                if (in_smem) {
                    det_add(&s_acc[e], &gv[e], pt[k][d], scale);
                    det_add(&s_acc[e], &gv[e], nt[k][d], scale);
                } else {
                    det_add(&av[e], &gv[e], pt[k][d], scale);
                    det_add(&av[e], &gv[e], nt[k][d], scale);
                }
            }
    }
    if (in_smem) {
        __syncthreads();
        for (int k = tid; k < V * 3; k += SN_THREADS) {
            const unsigned long long a = s_acc[k];
            if (a != 0ull) atomicAdd(&av[k], a);
        }
    }
}

// host-side checks shared by the backward entry points
static int sn_bwd_check(const float *verts, const int32_t *faces, const int32_t *face_idx, const float *uv,
                        const float *grad_normals, float *grad_verts, int64_t B, int64_t V, int64_t F, int64_t S,
                        const char *what) {
    PTK_REQUIRE(verts && faces && face_idx && uv && grad_normals && grad_verts, PTK_ERR_SHAPE, "%s: null pointer", what);
    PTK_REQUIRE(B > 0 && V > 0 && F > 0 && S > 0 && B <= 65535 && V < (1 << 28) && F < (1 << 28) && S < (1 << 28),
                PTK_ERR_SHAPE, "%s: bad sizes (B=%lld, V=%lld, F=%lld, S=%lld)", what, (long long)B, (long long)V,
                (long long)F, (long long)S);
    return PTK_OK;
}

}  // namespace ptk

using namespace ptk;

extern "C" int ptk_sample_normals_fwd(const float *verts, int64_t B, int64_t V, const int32_t *faces, int64_t F,
                                      const int32_t *face_idx, int64_t S, float *normals, ptk_stream_t stream) {
    PTK_NVTX("ptk_sample_normals_fwd");
    PTK_REQUIRE(verts && faces && face_idx && normals, PTK_ERR_SHAPE, "sample_normals_fwd: null pointer");
    PTK_REQUIRE(B > 0 && V > 0 && F > 0 && S > 0 && B <= 65535 && V < (1 << 28) && F < (1 << 28) && S < (1 << 28),
                PTK_ERR_SHAPE, "sample_normals_fwd: bad sizes (B=%lld, V=%lld, F=%lld, S=%lld)", (long long)B,
                (long long)V, (long long)F, (long long)S);
    launch_pdl(sample_normals_fwd_kernel, dim3((unsigned)ceil_div(S, SN_THREADS), (unsigned)B), dim3(SN_THREADS), 0,
               as_stream(stream), verts, (int)V, faces, (int)F, face_idx, (int)S, normals);
    PTK_CHECK_LAUNCH();
    return PTK_OK;
}

extern "C" int ptk_sample_normals_bwd(const float *verts, const int32_t *faces, const int32_t *face_idx, const float *uv,
                                      const float *grad_pts, const float *grad_normals, int64_t B, int64_t V, int64_t F,
                                      int64_t S, float *grad_verts, ptk_stream_t stream) {
    PTK_NVTX("ptk_sample_normals_bwd");
    int rc = sn_bwd_check(verts, faces, face_idx, uv, grad_normals, grad_verts, B, V, F, S, "sample_normals_bwd");
    if (rc) return rc;
    cudaStream_t st = as_stream(stream);
    PTK_CHECK_CUDA(cudaMemsetAsync(grad_verts, 0, sizeof(float) * (size_t)B * V * 3, st));
    launch_pdl(sample_normals_bwd_kernel, dim3((unsigned)ceil_div(S, SN_PER_CTA), (unsigned)B), dim3(SN_THREADS), 0, st,
               verts, faces, face_idx, uv, uv + (size_t)B * S, grad_pts, grad_normals, (int)V, (int)F, (int)S, grad_verts);
    PTK_CHECK_LAUNCH();
    return PTK_OK;
}

extern "C" size_t ptk_sample_normals_bwd_det_workspace_bytes(int64_t B, int64_t V) {
    if (B <= 0 || V <= 0) return 0;
    return det_workspace_bytes(B, V);
}

extern "C" int ptk_sample_normals_bwd_det(const float *verts, const int32_t *faces, const int32_t *face_idx,
                                          const float *uv, const float *grad_pts, const float *grad_normals, int64_t B,
                                          int64_t V, int64_t F, int64_t S, float *grad_verts, void *workspace,
                                          size_t workspace_bytes, ptk_stream_t stream) {
    PTK_NVTX("ptk_sample_normals_bwd_det");
    int rc = sn_bwd_check(verts, faces, face_idx, uv, grad_normals, grad_verts, B, V, F, S, "sample_normals_bwd_det");
    if (rc) return rc;
    rc = det_check_workspace(workspace, workspace_bytes, ptk_sample_normals_bwd_det_workspace_bytes(B, V),
                             "sample_normals_bwd_det");
    if (rc) return rc;
    cudaStream_t st = as_stream(stream);
    DetWs w;
    PTK_CHECK_CUDA(det_begin(workspace, B, V, st, w));
    const DetBound nb = det_bound_const(6LL * S + 1);
    const float *uu = uv, *vv = uv + (size_t)B * S;
    launch_pdl(sample_normals_bwd_det_max_kernel, dim3((unsigned)ceil_div(S > V ? S : V, SN_THREADS), (unsigned)B),
               dim3(SN_THREADS), 0, st, verts, faces, face_idx, uu, vv, grad_pts, grad_normals, (int)V, (int)F, (int)S,
               grad_verts, w.acc_a, w.mbits);
    PTK_CHECK_LAUNCH();
    launch_pdl(sample_normals_bwd_det_add_kernel, dim3((unsigned)ceil_div(S, SN_PER_CTA), (unsigned)B), dim3(SN_THREADS),
               0, st, verts, faces, face_idx, uu, vv, grad_pts, grad_normals, (int)V, (int)F, (int)S, grad_verts, w.acc_a,
               (const unsigned int *)w.mbits, nb);
    PTK_CHECK_LAUNCH();
    det_launch_convert<SN_THREADS>(w, nb, B, grad_verts, V, nullptr, 0, st);
    PTK_CHECK_LAUNCH();
    return PTK_OK;
}
