// Area-weighted surface point sampling for sm_100a.
//
// Replaces the body of utils.batch_sample (pterotactyl/utility/utils.py:152-187):
//   mesh_face_areas_normals (utils.py:164) + NaN guards (165-168) + Tensor.multinomial (170) +
//   _rand_barycentric_coords (179) + barycentric interpolation (182-185)  ~ 25 ATen launches,
// with two kernels:
//   sample_prepare_kernel : per mesh, face areas -> max -> 32.32 fixed-point weights -> inclusive
//                           uint64 prefix sum (order independent => bit-exact by construction)
//   sample_points_kernel  : per sample, 128-bit multiply + binary search (prefix sums staged in
//                           shared memory) + vertex gather + barycentric interpolation with
//                           individually rounded ops in the reference's order.
// The arithmetic is defined in oracle/ptk_oracle.c (orc_face_cumweights / orc_sample_fwd); this file
// must match it bit for bit.
#include "det_accum.cuh"

namespace ptk {

constexpr int SP_THREADS = 256;
constexpr int SP_SMEM_FACES = 4096;  // prefix sums of up to 4096 faces live in shared memory (32 KB)

__device__ __forceinline__ float face_area_rn(const float *__restrict__ v0,
                                              const float *__restrict__ v1,
                                              const float *__restrict__ v2) {
    float ax = __fsub_rn(v1[0], v0[0]), ay = __fsub_rn(v1[1], v0[1]), az = __fsub_rn(v1[2], v0[2]);
    float bx = __fsub_rn(v2[0], v0[0]), by = __fsub_rn(v2[1], v0[1]), bz = __fsub_rn(v2[2], v0[2]);
    float cx = __fsub_rn(__fmul_rn(ay, bz), __fmul_rn(az, by));
    float cy = __fsub_rn(__fmul_rn(az, bx), __fmul_rn(ax, bz));
    float cz = __fsub_rn(__fmul_rn(ax, by), __fmul_rn(ay, bx));
    float n2 = __fadd_rn(__fadd_rn(__fmul_rn(cx, cx), __fmul_rn(cy, cy)), __fmul_rn(cz, cz));
    return __fmul_rn(__fsqrt_rn(n2), 0.5f);
}

__device__ __forceinline__ unsigned long long face_weight(float a, float amax) {
    if (amax == 0.0f) return 1ull;
    if (isinf(amax)) return isinf(a) ? 1ull : 0ull;
    double q = __dmul_rn(__ddiv_rn((double)a, (double)amax), 4294967296.0);
    return (unsigned long long)q;  // truncation, q in [0, 2^32]
}

// grid = B, block = SP_THREADS.  cum (B,F) uint64 inclusive prefix sums of the integer weights.
__global__ void __launch_bounds__(SP_THREADS)
sample_prepare_kernel(const float *__restrict__ verts, int V, const int32_t *__restrict__ faces, int F,
                      unsigned long long *__restrict__ cum, float *__restrict__ areas) {
    pdl_wait();  // launched with programmatic stream serialization (ptk_common.cuh)
    const int b = blockIdx.x;
    const int tid = threadIdx.x;
    const float *vb = verts + (size_t)b * V * 3;
    float *ab = areas + (size_t)b * F;
    unsigned long long *cb = cum + (size_t)b * F;
    __shared__ float s_red[SP_THREADS / 32];
    __shared__ unsigned long long s_scan[SP_THREADS / 32];
    __shared__ float s_amax;

    // pass 1: areas (NaN -> 0) and their maximum
    float amax = 0.0f;
    for (int f = tid; f < F; f += SP_THREADS) {
        int i0 = faces[f * 3 + 0], i1 = faces[f * 3 + 1], i2 = faces[f * 3 + 2];
        float a = face_area_rn(vb + (size_t)i0 * 3, vb + (size_t)i1 * 3, vb + (size_t)i2 * 3);
        a = (a != a) ? 0.0f : a;
        ab[f] = a;
        amax = fmaxf(amax, a);
    }
    amax = warp_max(amax);
    if ((tid & 31) == 0) s_red[tid >> 5] = amax;
    __syncthreads();
    if (tid == 0) {
        float m = s_red[0];
        for (int w = 1; w < SP_THREADS / 32; ++w) m = fmaxf(m, s_red[w]);
        s_amax = m;
    }
    __syncthreads();
    amax = s_amax;

    // pass 2: contiguous segment per thread -> segment sums -> block scan -> write-out
    const int seg = (F + SP_THREADS - 1) / SP_THREADS;
    const int f0 = tid * seg;
    const int f1 = min(F, f0 + seg);
    unsigned long long local = 0;
    for (int f = f0; f < f1; ++f) local += face_weight(ab[f], amax);
    // inclusive warp scan of `local`
    unsigned long long incl = local;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        unsigned long long up = __shfl_up_sync(0xffffffffu, incl, o);
        if ((tid & 31) >= o) incl += up;
    }
    if ((tid & 31) == 31) s_scan[tid >> 5] = incl;
    __syncthreads();
    unsigned long long base = 0;
    for (int w = 0; w < (tid >> 5); ++w) base += s_scan[w];
    unsigned long long run = base + incl - local;  // exclusive prefix of this thread's segment
    for (int f = f0; f < f1; ++f) {
        run += face_weight(ab[f], amax);
        cb[f] = run;
    }
}

// grid = (ceil(S / SP_THREADS), B)
__global__ void __launch_bounds__(SP_THREADS)
sample_points_kernel(const float *__restrict__ verts, int V, const int32_t *__restrict__ faces, int F,
                     const unsigned long long *__restrict__ cum, const float *__restrict__ u_face,
                     const float *__restrict__ uu, const float *__restrict__ vv, int S,
                     float *__restrict__ pts, int32_t *__restrict__ face_idx) {
    pdl_wait();  // launched with programmatic stream serialization (ptk_common.cuh)
    const int b = blockIdx.y;
    const int tid = threadIdx.x;
    const unsigned long long *cb = cum + (size_t)b * F;
    __shared__ unsigned long long s_cum[SP_SMEM_FACES];
    const bool given = u_face == nullptr;  // the caller drew the faces (face_idx is an input): interpolation only
    const bool in_smem = !given && F <= SP_SMEM_FACES;
    if (in_smem) {
        for (int f = tid; f < F; f += SP_THREADS) s_cum[f] = cb[f];
        __syncthreads();
    }
    const int s = blockIdx.x * SP_THREADS + tid;
    if (s >= S) return;
    const size_t o = (size_t)b * S + s;

    int f;
    if (given) {
        f = min(max(face_idx[o], 0), F - 1);  // an out-of-range id never reads outside the face list
    } else {
        // face pick: r = (floor(u * 2^24) * total) >> 24 ; first f with cum[f] > r
        const float sc = __fmul_rn(u_face[o], 16777216.0f);
        unsigned long long t = sc >= 16777215.0f ? 16777215ull : (sc > 0.0f ? (unsigned long long)sc : 0ull);
        const unsigned long long total = in_smem ? s_cum[F - 1] : cb[F - 1];
        // (t * total) >> 24  ==  hi64((t << 40) * total)
        const unsigned long long r = __umul64hi(t << 40, total);
        int lo = 0, hi = F - 1;
        while (lo < hi) {
            int mid = (lo + hi) >> 1;
            unsigned long long c = in_smem ? s_cum[mid] : cb[mid];
            if (c > r)
                hi = mid;
            else
                lo = mid + 1;
        }
        f = lo;
    }
    const float *vb = verts + (size_t)b * V * 3;
    const float *A = vb + (size_t)faces[f * 3 + 0] * 3;
    const float *Bv = vb + (size_t)faces[f * 3 + 1] * 3;
    const float *Cv = vb + (size_t)faces[f * 3 + 2] * 3;
    const float rt = __fsqrt_rn(uu[o]);
    const float v = vv[o];
    const float w0 = __fsub_rn(1.0f, rt);
    const float w1 = __fmul_rn(rt, __fsub_rn(1.0f, v));
    const float w2 = __fmul_rn(rt, v);
#pragma unroll
    for (int d = 0; d < 3; ++d) {
        float t0 = __fmul_rn(w0, A[d]);
        float t1 = __fmul_rn(w1, Bv[d]);
        float t2 = __fmul_rn(w2, Cv[d]);
        pts[o * 3 + d] = __fadd_rn(__fadd_rn(t0, t1), t2);
    }
    face_idx[o] = f;
}

// grad_verts[b, faces[f,k]] += w_k * grad_pts[b,s]   (grad_verts zeroed by the caller below)
// grid = (ceil(S / SP_THREADS), B).  Accumulates in shared memory when the mesh fits, then one
// global RED per touched vertex component.
constexpr int SB_SMEM_VERTS = 4096;  // 4096 * 3 floats = 48 KB

__global__ void __launch_bounds__(SP_THREADS)
sample_bwd_kernel(const float *__restrict__ grad_pts, const int32_t *__restrict__ face_idx,
                  const float *__restrict__ uu, const float *__restrict__ vv,
                  const int32_t *__restrict__ faces, int V, int S, int samples_per_cta,
                  float *__restrict__ grad_verts) {
    pdl_wait();  // launched with programmatic stream serialization (ptk_common.cuh)
    const int b = blockIdx.y;
    const int tid = threadIdx.x;
    __shared__ float s_acc[SB_SMEM_VERTS * 3];
    const bool in_smem = V <= SB_SMEM_VERTS;
    if (in_smem) {
        for (int k = tid; k < V * 3; k += SP_THREADS) s_acc[k] = 0.0f;
        __syncthreads();
    }
    float *gv = grad_verts + (size_t)b * V * 3;
    const int s_begin = blockIdx.x * samples_per_cta;
    const int s_end = min(S, s_begin + samples_per_cta);
    for (int s = s_begin + tid; s < s_end; s += SP_THREADS) {
        const size_t o = (size_t)b * S + s;
        const int f = face_idx[o];
        const float rt = __fsqrt_rn(uu[o]);
        const float v = vv[o];
        const float w[3] = {__fsub_rn(1.0f, rt), __fmul_rn(rt, __fsub_rn(1.0f, v)), __fmul_rn(rt, v)};
        const float g[3] = {grad_pts[o * 3 + 0], grad_pts[o * 3 + 1], grad_pts[o * 3 + 2]};
#pragma unroll
        for (int k = 0; k < 3; ++k) {
            const int vi = faces[f * 3 + k];
#pragma unroll
            for (int d = 0; d < 3; ++d) {
                float c = __fmul_rn(w[k], g[d]);
                if (in_smem)
                    atomicAdd(&s_acc[vi * 3 + d], c);
                else
                    atomicAdd(&gv[(size_t)vi * 3 + d], c);
            }
        }
    }
    if (in_smem) {
        __syncthreads();
        for (int k = tid; k < V * 3; k += SP_THREADS) {
            float a = s_acc[k];
            if (a != 0.0f) atomicAdd(&gv[k], a);
        }
    }
}

// Deterministic backward (ptk_sample_bwd_det, scheme in det_accum.cuh).  The terms are c = w_k * g_d with the
// arithmetic of sample_bwd_kernel; a vertex receives at most 3 S of them (a degenerate face may list it twice).
// phase 1, grid = (ceil(max(S, V) / SP_THREADS), B): M_b (atomicMax into mbits[b], zeroed by the caller); zero the
// accumulators and grad_verts
__device__ __forceinline__ void sample_det_weights(const float *__restrict__ uu, const float *__restrict__ vv, size_t o,
                                                   float w[3]) {
    const float rt = __fsqrt_rn(uu[o]);
    const float v = vv[o];
    w[0] = __fsub_rn(1.0f, rt);
    w[1] = __fmul_rn(rt, __fsub_rn(1.0f, v));
    w[2] = __fmul_rn(rt, v);
}

__global__ void __launch_bounds__(SP_THREADS)
sample_bwd_det_terms_kernel(const float *__restrict__ grad_pts, const float *__restrict__ uu, const float *__restrict__ vv,
                            int V, int S, float *__restrict__ grad_verts, unsigned long long *__restrict__ acc,
                            unsigned int *__restrict__ mbits) {
    pdl_wait();
    const int b = blockIdx.y;
    const int i = blockIdx.x * SP_THREADS + threadIdx.x;
    float m = 0.0f;
    if (i < S) {
        const size_t o = (size_t)b * S + i;
        float w[3];
        sample_det_weights(uu, vv, o, w);
#pragma unroll
        for (int k = 0; k < 3; ++k)
#pragma unroll
            for (int d = 0; d < 3; ++d) m = fmaxf(m, det_abs_finite(__fmul_rn(w[k], grad_pts[o * 3 + d])));
    }
    if (i < V) det_zero_row(acc, grad_verts, (size_t)b * V + i);
    det_block_max<SP_THREADS>(m, mbits + b);
}

// phase 2, grid = (ceil(S / samples_per_cta), B): quantise and add.  Meshes of up to SBD_SMEM_VERTS vertices are
// accumulated in shared memory first (exact as well), then one global 64-bit reduction per touched component.
constexpr int SBD_SMEM_VERTS = 2048;  // 2048 * 3 int64 = 48 KB

__global__ void __launch_bounds__(SP_THREADS)
sample_bwd_det_reduce_kernel(const float *__restrict__ grad_pts, const int32_t *__restrict__ face_idx,
                             const float *__restrict__ uu, const float *__restrict__ vv, const int32_t *__restrict__ faces,
                             int V, int S, int samples_per_cta, float *__restrict__ grad_verts,
                             unsigned long long *__restrict__ acc, const unsigned int *__restrict__ mbits, DetBound nb) {
    pdl_wait();
    const int b = blockIdx.y;
    const int tid = threadIdx.x;
    __shared__ unsigned long long s_acc[SBD_SMEM_VERTS * 3];
    const bool in_smem = V <= SBD_SMEM_VERTS;
    if (in_smem) {
        for (int k = tid; k < V * 3; k += SP_THREADS) s_acc[k] = 0ull;
        __syncthreads();
    }
    const double scale = det_scale(mbits, nb, b);
    float *gv = grad_verts + (size_t)b * V * 3;
    unsigned long long *av = acc + (size_t)b * V * 3;
    const int s_begin = blockIdx.x * samples_per_cta;
    const int s_end = min(S, s_begin + samples_per_cta);
    for (int s = s_begin + tid; s < s_end; s += SP_THREADS) {
        const size_t o = (size_t)b * S + s;
        const int f = face_idx[o];
        float w[3];
        sample_det_weights(uu, vv, o, w);
        const float g[3] = {grad_pts[o * 3 + 0], grad_pts[o * 3 + 1], grad_pts[o * 3 + 2]};
#pragma unroll
        for (int k = 0; k < 3; ++k) {
            const int vi = faces[f * 3 + k];
#pragma unroll
            for (int d = 0; d < 3; ++d) {
                const float c = __fmul_rn(w[k], g[d]);
                if (in_smem)
                    det_add(&s_acc[vi * 3 + d], &gv[(size_t)vi * 3 + d], c, scale);
                else
                    det_add(&av[(size_t)vi * 3 + d], &gv[(size_t)vi * 3 + d], c, scale);
            }
        }
    }
    if (in_smem) {
        __syncthreads();
        for (int k = tid; k < V * 3; k += SP_THREADS) {
            const unsigned long long a = s_acc[k];
            if (a != 0ull) atomicAdd(&av[k], a);
        }
    }
}

// pytorch3d.ops.mesh_face_areas_normals drop-in (packed verts (V,3), int64 faces (F,3)): areas (F) and
// unit normals (F,3) with the 1e-6 clamp of PyTorch3D's face_areas_normals kernel.
__global__ void face_areas_normals_kernel(const float *__restrict__ verts, const long long *__restrict__ faces,
                                          long long F, float *__restrict__ areas,
                                          float *__restrict__ normals) {
    const long long f = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (f >= F) return;
    const float *v0 = verts + faces[f * 3 + 0] * 3, *v1 = verts + faces[f * 3 + 1] * 3,
                *v2 = verts + faces[f * 3 + 2] * 3;
    float ax = __fsub_rn(v1[0], v0[0]), ay = __fsub_rn(v1[1], v0[1]), az = __fsub_rn(v1[2], v0[2]);
    float bx = __fsub_rn(v2[0], v0[0]), by = __fsub_rn(v2[1], v0[1]), bz = __fsub_rn(v2[2], v0[2]);
    float cx = __fsub_rn(__fmul_rn(ay, bz), __fmul_rn(az, by));
    float cy = __fsub_rn(__fmul_rn(az, bx), __fmul_rn(ax, bz));
    float cz = __fsub_rn(__fmul_rn(ax, by), __fmul_rn(ay, bx));
    float n = __fsqrt_rn(__fadd_rn(__fadd_rn(__fmul_rn(cx, cx), __fmul_rn(cy, cy)), __fmul_rn(cz, cz)));
    areas[f] = __fmul_rn(n, 0.5f);
    if (normals) {
        float inv = n < 1e-6f ? 1e-6f : n;
        normals[f * 3 + 0] = cx / inv;
        normals[f * 3 + 1] = cy / inv;
        normals[f * 3 + 2] = cz / inv;
    }
}

// areas (B,F) of a batch of meshes sharing one int32 face list: the quantity utils.batch_sample normalises and hands to
// Tensor.multinomial (utils.py:163-170).  Same individually rounded arithmetic as above; NaN areas are kept (the
// reference zeroes them itself, utils.py:165).
__global__ void mesh_face_areas_kernel(const float *__restrict__ verts, int V, const int32_t *__restrict__ faces,
                                       int F, float *__restrict__ areas) {
    const int f = blockIdx.x * blockDim.x + threadIdx.x;
    if (f >= F) return;
    const float *vb = verts + (size_t)blockIdx.y * V * 3;
    const int i0 = faces[f * 3 + 0], i1 = faces[f * 3 + 1], i2 = faces[f * 3 + 2];
    areas[(size_t)blockIdx.y * F + f] = face_area_rn(vb + (size_t)i0 * 3, vb + (size_t)i1 * 3, vb + (size_t)i2 * 3);
}

}  // namespace ptk

using namespace ptk;

extern "C" int ptk_mesh_face_areas(const float *verts, int64_t B, int64_t V, const int32_t *faces, int64_t F,
                                   float *areas, ptk_stream_t stream) {
    PTK_REQUIRE(verts && faces && areas, PTK_ERR_SHAPE, "mesh_face_areas: null pointer");
    PTK_REQUIRE(B > 0 && V > 0 && F > 0 && B <= 65535 && F < (1 << 28) && V < (1 << 28), PTK_ERR_SHAPE,
                "mesh_face_areas: bad sizes (B=%lld, V=%lld, F=%lld)", (long long)B, (long long)V, (long long)F);
    mesh_face_areas_kernel<<<dim3((unsigned)ceil_div(F, 256), (unsigned)B), 256, 0, as_stream(stream)>>>(
        verts, (int)V, faces, (int)F, areas);
    PTK_CHECK_LAUNCH();
    return PTK_OK;
}

extern "C" int ptk_face_areas_normals(const float *verts, int64_t V, const int64_t *faces, int64_t F,
                                      float *areas, float *normals, ptk_stream_t stream) {
    PTK_REQUIRE(verts && faces && areas, PTK_ERR_SHAPE, "face_areas_normals: null pointer");
    PTK_REQUIRE(V > 0 && F >= 0, PTK_ERR_SHAPE, "face_areas_normals: bad sizes");
    if (F == 0) return PTK_OK;
    face_areas_normals_kernel<<<(unsigned)ceil_div(F, 256), 256, 0, as_stream(stream)>>>(
        verts, (const long long *)faces, (long long)F, areas, normals);
    PTK_CHECK_LAUNCH();
    return PTK_OK;
}

extern "C" size_t ptk_sample_workspace_bytes(int64_t B, int64_t F) {
    if (B <= 0 || F <= 0) return 0;
    // uint64 prefix sums + fp32 areas
    return (size_t)B * (size_t)F * (sizeof(unsigned long long) + sizeof(float));
}

extern "C" int ptk_sample_fwd(const float *verts, int64_t B, int64_t V, const int32_t *faces,
                              int64_t F, const float *u_face, const float *uv, int64_t S, float *pts,
                              int32_t *face_idx, void *workspace, size_t workspace_bytes,
                              ptk_stream_t stream) {
    PTK_NVTX("ptk_sample_fwd");
    PTK_REQUIRE(verts && faces && uv && pts && face_idx, PTK_ERR_SHAPE, "sample_fwd: null pointer");
    PTK_REQUIRE(B > 0 && V > 0 && F > 0 && S > 0, PTK_ERR_SHAPE,
                "sample_fwd: empty input (B=%lld, V=%lld, F=%lld, S=%lld)", (long long)B, (long long)V,
                (long long)F, (long long)S);
    PTK_REQUIRE(B <= 65535 && F < (1 << 28) && V < (1 << 28), PTK_ERR_SHAPE, "sample_fwd: size out of range");
    cudaStream_t st = as_stream(stream);
    unsigned long long *cum = nullptr;
    if (u_face) {  // NULL: the caller supplies face_idx (drawn by its own RNG), only the interpolation runs
        PTK_REQUIRE(workspace && workspace_bytes >= ptk_sample_workspace_bytes(B, F), PTK_ERR_WORKSPACE,
                    "sample_fwd: workspace too small");
        cum = reinterpret_cast<unsigned long long *>(workspace);
        auto *areas = reinterpret_cast<float *>(cum + (size_t)B * F);
        launch_pdl(sample_prepare_kernel, dim3((unsigned)B), dim3(SP_THREADS), 0, st, verts, (int)V, faces, (int)F, cum, areas);
        PTK_CHECK_LAUNCH();
    }
    dim3 grid((unsigned)ceil_div(S, SP_THREADS), (unsigned)B);
    launch_pdl(sample_points_kernel, grid, dim3(SP_THREADS), 0, st, verts, (int)V, faces, (int)F, cum, u_face, uv,
               uv + (size_t)B * S, (int)S, pts, face_idx);
    PTK_CHECK_LAUNCH();
    return PTK_OK;
}

extern "C" int ptk_sample_bwd(const float *grad_pts, const int32_t *face_idx, const float *uv,
                              const int32_t *faces, int64_t B, int64_t V, int64_t F, int64_t S,
                              float *grad_verts, ptk_stream_t stream) {
    PTK_NVTX("ptk_sample_bwd");
    PTK_REQUIRE(grad_pts && face_idx && uv && faces && grad_verts, PTK_ERR_SHAPE, "sample_bwd: null pointer");
    PTK_REQUIRE(B > 0 && V > 0 && F > 0 && S > 0 && B <= 65535, PTK_ERR_SHAPE, "sample_bwd: bad sizes");
    cudaStream_t st = as_stream(stream);
    PTK_CHECK_CUDA(cudaMemsetAsync(grad_verts, 0, sizeof(float) * (size_t)B * V * 3, st));
    const int per_cta = 2048;
    dim3 grid((unsigned)ceil_div(S, per_cta), (unsigned)B);
    launch_pdl(sample_bwd_kernel, grid, dim3(SP_THREADS), 0, st, grad_pts, face_idx, uv, uv + (size_t)B * S, faces, (int)V,
               (int)S, per_cta, grad_verts);
    PTK_CHECK_LAUNCH();
    return PTK_OK;
}

extern "C" size_t ptk_sample_bwd_det_workspace_bytes(int64_t B, int64_t V) {
    if (B <= 0 || V <= 0) return 0;
    return det_workspace_bytes(B, V);
}

extern "C" int ptk_sample_bwd_det(const float *grad_pts, const int32_t *face_idx, const float *uv, const int32_t *faces,
                                  int64_t B, int64_t V, int64_t F, int64_t S, float *grad_verts, void *workspace,
                                  size_t workspace_bytes, ptk_stream_t stream) {
    PTK_NVTX("ptk_sample_bwd_det");
    PTK_REQUIRE(grad_pts && face_idx && uv && faces && grad_verts, PTK_ERR_SHAPE, "sample_bwd_det: null pointer");
    PTK_REQUIRE(B > 0 && V > 0 && F > 0 && S > 0 && B <= 65535 && V < (1 << 28) && S < (1 << 28), PTK_ERR_SHAPE,
                "sample_bwd_det: bad sizes");
    int rc = det_check_workspace(workspace, workspace_bytes, ptk_sample_bwd_det_workspace_bytes(B, V), "sample_bwd_det");
    if (rc) return rc;
    cudaStream_t st = as_stream(stream);
    DetWs w;
    PTK_CHECK_CUDA(det_begin(workspace, B, V, st, w));
    const DetBound nb = det_bound_const(3LL * S + 1);
    const float *uu = uv, *vv = uv + (size_t)B * S;
    launch_pdl(sample_bwd_det_terms_kernel, dim3((unsigned)ceil_div(S > V ? S : V, SP_THREADS), (unsigned)B), dim3(SP_THREADS),
               0, st, grad_pts, uu, vv, (int)V, (int)S, grad_verts, w.acc_a, w.mbits);
    PTK_CHECK_LAUNCH();
    const int per_cta = 2048;
    launch_pdl(sample_bwd_det_reduce_kernel, dim3((unsigned)ceil_div(S, per_cta), (unsigned)B), dim3(SP_THREADS), 0, st,
               grad_pts, face_idx, uu, vv, faces, (int)V, (int)S, per_cta, grad_verts, w.acc_a, (const unsigned int *)w.mbits,
               nb);
    PTK_CHECK_LAUNCH();
    det_launch_convert<SP_THREADS>(w, nb, B, grad_verts, V, nullptr, 0, st);
    PTK_CHECK_LAUNCH();
    return PTK_OK;
}
