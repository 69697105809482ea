// Chamfer normal term for sm_100a: the cham_normals of PyTorch3D 0.5.0's chamfer_distance(x_normals=, y_normals=),
// on the nearest-neighbour indices of ptk_chamfer_fwd_lengths.  Contract in include/ptk.h (ptk_chamfer_normals_fwd),
// design and cost in DESIGN.md K1d.
//
// For a valid query i < lq of pair b with j = idx[b,i], a = its normal and n = normal j of the other cloud:
//     c = sum_k (a_k / max(|a|, 1e-6)) * (n_k / max(|n|, 1e-6))      (torch's F.cosine_similarity, eps = 1e-6)
//     term = 1 - |c|
// A valid query whose target cloud is empty reads PyTorch3D's zero-filled gathered normal (n = 0: c = 0, term 1);
// padded queries have term 0.  The forward is memory-bound (a query reads its normal, its idx and one gathered normal)
// and reduces each pair in the fixed order of chamfer_finalize_kernel (fin_splits of the pair's own lengths, slice
// partials added in slice order).  The backward splits a term's gradient into an "own" part on the query's normal row
// and a "near" part on the gathered normal's row, recomputing c from the normals.
#include "pair_bwd.cuh"

namespace ptk {

constexpr float CN_EPS = 1e-6f;  // F.cosine_similarity's default eps, clamped per norm

__device__ __forceinline__ void load_normal(const float *__restrict__ p, int i, float v[3]) {
    v[0] = p[i * 3 + 0];
    v[1] = p[i * 3 + 1];
    v[2] = p[i * 3 + 2];
}

// c of the query normal a and the gathered normal n, torch's order: both divided by their clamped norms, then the
// products summed.  ra / rn: the unclamped norms, ua / un: the divided vectors.
__device__ __forceinline__ float normal_cos(const float a[3], const float n[3], float &ra, float &rn, float ua[3],
                                            float un[3]) {
    ra = sqrtf(a[0] * a[0] + a[1] * a[1] + a[2] * a[2]);
    rn = sqrtf(n[0] * n[0] + n[1] * n[1] + n[2] * n[2]);
    const float na = fmaxf(ra, CN_EPS), nn = fmaxf(rn, CN_EPS);
#pragma unroll
    for (int k = 0; k < 3; ++k) {
        ua[k] = a[k] / na;
        un[k] = n[k] / nn;
    }
    return ua[0] * un[0] + ua[1] * un[1] + ua[2] * un[2];
}

// term of valid query i (qn / tn: the query and target clouds' normals of the pair); Lt = 0 gathers the zero normal
__device__ __forceinline__ float normal_term(const float *__restrict__ qn, const float *__restrict__ tn,
                                             const int32_t *__restrict__ idx, int i, int Lt) {
    float a[3], n[3] = {0.0f, 0.0f, 0.0f}, ra, rn, ua[3], un[3];
    load_normal(qn, i, a);
    if (Lt > 0) load_normal(tn, idx[i], n);
    return 1.0f - fabsf(normal_cos(a, n, ra, rn, ua, un));
}

// Forward, grid = (B, nsplit = fin_splits(P1, P2)), block = 512: CTA (b, s) sums slice s of both directions' terms of
// pair b (slices of the pair's own lengths; CTAs past that count only zero-fill padded term entries).  Unsliced it
// writes cham_n[b], otherwise its two partial sums, which chamfer_normals_sum_kernel adds in slice order.
__global__ void __launch_bounds__(512)
chamfer_normals_fwd_kernel(const float *__restrict__ xn, const float *__restrict__ yn, const int32_t *__restrict__ idx_x,
                           const int32_t *__restrict__ idx_y, int P1, int P2, const int64_t *__restrict__ len_x,
                           const int64_t *__restrict__ len_y, int mean, float *__restrict__ term_x,
                           float *__restrict__ term_y, float *__restrict__ cham_n, float *__restrict__ partial) {
    pdl_wait();
    const int b = blockIdx.x, sp = blockIdx.y, nsp = gridDim.y;
    const int tid = threadIdx.x;
    const int L1 = pair_len(len_x, b, P1), L2 = pair_len(len_y, b, P2);
    const int nv = fin_splits(L1, L2);
    __shared__ float red[16];
    float sum[2] = {0.f, 0.f};
#pragma unroll
    for (int dir = 0; dir < 2; ++dir) {
        const int P = dir == 0 ? P1 : P2, Pt = dir == 0 ? P2 : P1;
        const int L = dir == 0 ? L1 : L2, Lt = dir == 0 ? L2 : L1;
        const float *qn = (dir == 0 ? xn : yn) + (size_t)b * P * 3;
        const float *tn = (dir == 0 ? yn : xn) + (size_t)b * Pt * 3;
        const int32_t *idx = (dir == 0 ? idx_x : idx_y) + (size_t)b * P;
        float *term = dir == 0 ? term_x : term_y;
        float acc = 0.f;
        if (sp < nv) {
            const int len = (int)(((long long)L + nv - 1) / nv), i0 = sp * len, i1 = min(L, i0 + len);
#pragma unroll 4
            for (int i = i0 + tid; i < i1; i += 512) {
                const float t = normal_term(qn, tn, idx, i, Lt);
                if (term) term[(size_t)b * P + i] = t;
                acc += t;
            }
        }
        if (term) {
            const int plen = (P - L + nsp - 1) / nsp, p0 = L + sp * plen, p1 = min(P, p0 + plen);
            for (int i = p0 + tid; i < p1; i += 512) term[(size_t)b * P + i] = 0.f;
        }
        acc = warp_sum(acc);
        __syncthreads();
        if ((tid & 31) == 0) red[tid >> 5] = acc;
        __syncthreads();
        if (tid < 32) {
            float v = tid < 16 ? red[tid] : 0.f;
            v = warp_sum(v);
            if (tid == 0) sum[dir] = v;
        }
    }
    if (tid == 0) {
        if (nsp == 1) {
            cham_n[b] = chamfer_reduce(sum[0], sum[1], L1, L2, mean);
        } else if (sp < nv) {
            partial[((size_t)b * nsp + sp) * 2 + 0] = sum[0];
            partial[((size_t)b * nsp + sp) * 2 + 1] = sum[1];
        }
    }
}

// grid = ceil(B / 128), block = 128: cham_n[b] from the pair's slice partials, in slice order
__global__ void __launch_bounds__(128)
chamfer_normals_sum_kernel(const float *__restrict__ partial, int B, int nsp, int P1, int P2,
                           const int64_t *__restrict__ len_x, const int64_t *__restrict__ len_y, int mean,
                           float *__restrict__ cham_n) {
    pdl_wait();
    const int b = blockIdx.x * 128 + threadIdx.x;
    if (b >= B) return;
    const int L1 = pair_len(len_x, b, P1), L2 = pair_len(len_y, b, P2);
    const int nv = fin_splits(L1, L2);
    float sx = 0.f, sy = 0.f;
    for (int s = 0; s < nv; ++s) {
        sx += partial[((size_t)b * nsp + s) * 2 + 0];
        sy += partial[((size_t)b * nsp + s) * 2 + 1];
    }
    cham_n[b] = chamfer_reduce(sx, sy, L1, L2, mean);
}

// The gradient of query i's term under the upstream gradient g of its pair, torch's autograd of the forward formula:
//   d term / dc = -sign(c) (sign(0) = 0), scaled by s = g / lq (mean) or g (sum);
//   dc/da = (n / |n|_c - c * a / |a|) / |a|_c  -> own[]  (a / |a| = 0 at a = 0: the gradient of torch's norm there)
//   dc/dn = (a / |a|_c - c * n / |n|) / |n|_c  -> near[] (onto the gathered row j)
// false: no parts (padded query, or an empty target cloud: the gathered normal is PyTorch3D's constant zero fill).
__device__ __forceinline__ bool normal_parts(const float *__restrict__ qn, const float *__restrict__ tn,
                                             const int32_t *__restrict__ idx, float g, int i, int Lq, int Lt, int mean,
                                             int &j, float own[3], float near[3]) {
    if (i >= Lq || Lt <= 0) return false;
    j = idx[i];
    float a[3], n[3], ra, rn, ua[3], un[3];
    load_normal(qn, i, a);
    load_normal(tn, j, n);
    const float c = normal_cos(a, n, ra, rn, ua, un);
    const float s = mean ? g / (float)Lq : g;
    const float k = -s * (c > 0.0f ? 1.0f : (c < 0.0f ? -1.0f : 0.0f));
    const float na = fmaxf(ra, CN_EPS), nn = fmaxf(rn, CN_EPS);
#pragma unroll
    for (int d = 0; d < 3; ++d) {
        const float ha = ra > 0.0f ? a[d] / ra : 0.0f, hn = rn > 0.0f ? n[d] / rn : 0.0f;
        own[d] = k * ((un[d] - c * ha) / na);
        near[d] = k * ((ua[d] - c * hn) / nn);
    }
    return true;
}

// host-side checks shared by the three entry points
static int normals_check(const float *xn, const float *yn, const int32_t *idx_x, const int32_t *idx_y, int64_t B,
                         int64_t P1, int64_t P2, int reduction, const char *what) {
    PTK_REQUIRE(xn && yn && idx_x && idx_y, PTK_ERR_SHAPE, "%s: null normals / idx pointer", what);
    int rc = check_clouds(xn, yn, B, P1, P2);
    if (rc) return rc;
    PTK_REQUIRE(reduction == PTK_REDUCE_MEAN || reduction == PTK_REDUCE_SUM, PTK_ERR_SHAPE, "%s: unknown point reduction %d",
                what, reduction);
    PTK_REQUIRE(B <= 65535, PTK_ERR_SHAPE, "%s: batch too large", what);
    return PTK_OK;
}

}  // namespace ptk

using namespace ptk;

// slice partials: two floats per slice of every pair, only when the clouds are sliced (more than FIN_SLICE points)
extern "C" size_t ptk_chamfer_normals_workspace_bytes(int64_t B, int64_t P1, int64_t P2) {
    if (B <= 0 || P1 <= 0 || P2 <= 0) return 0;
    const int nsp = fin_splits(P1, P2);
    return nsp > 1 ? 8 * (size_t)B * nsp : 0;
}

extern "C" int ptk_chamfer_normals_fwd(const float *x_normals, const float *y_normals, const int64_t *len_x,
                                       const int64_t *len_y, const int32_t *idx_x, const int32_t *idx_y, int64_t B,
                                       int64_t P1, int64_t P2, int reduction, float *term_x, float *term_y,
                                       float *cham_normals, void *workspace, size_t workspace_bytes, ptk_stream_t stream) {
    PTK_NVTX("ptk_chamfer_normals_fwd");
    int rc = normals_check(x_normals, y_normals, idx_x, idx_y, B, P1, P2, reduction, "chamfer_normals_fwd");
    if (rc) return rc;
    PTK_REQUIRE(cham_normals, PTK_ERR_SHAPE, "chamfer_normals_fwd: null cham_normals pointer");
    const size_t need = ptk_chamfer_normals_workspace_bytes(B, P1, P2);
    PTK_REQUIRE(workspace_bytes >= need && (need == 0 || workspace), PTK_ERR_WORKSPACE,
                "chamfer_normals_fwd: workspace too small (%zu < %zu)", workspace_bytes, need);
    PTK_REQUIRE((reinterpret_cast<uintptr_t>(workspace) & 15) == 0, PTK_ERR_ALIGN,
                "chamfer_normals_fwd: workspace must be 16-byte aligned");
    cudaStream_t st = as_stream(stream);
    const int nsp = fin_splits(P1, P2);
    const int mean = reduction == PTK_REDUCE_MEAN ? 1 : 0;
    float *partial = reinterpret_cast<float *>(workspace);
    launch_pdl(chamfer_normals_fwd_kernel, dim3((unsigned)B, (unsigned)nsp), dim3(512), 0, st, x_normals, y_normals, idx_x,
               idx_y, (int)P1, (int)P2, len_x, len_y, mean, term_x, term_y, cham_normals, partial);
    PTK_CHECK_LAUNCH();
    if (nsp > 1) {
        launch_pdl(chamfer_normals_sum_kernel, dim3((unsigned)ceil_div(B, (int64_t)128)), dim3(128), 0, st,
                   (const float *)partial, (int)B, nsp, (int)P1, (int)P2, len_x, len_y, mean, cham_normals);
        PTK_CHECK_LAUNCH();
    }
    return PTK_OK;
}

extern "C" int ptk_chamfer_normals_bwd(const float *x_normals, const float *y_normals, const int64_t *len_x,
                                       const int64_t *len_y, const int32_t *idx_x, const int32_t *idx_y,
                                       const float *grad_cham_normals, int64_t B, int64_t P1, int64_t P2, int reduction,
                                       float *grad_xn, float *grad_yn, ptk_stream_t stream) {
    PTK_NVTX("ptk_chamfer_normals_bwd");
    int rc = normals_check(x_normals, y_normals, idx_x, idx_y, B, P1, P2, reduction, "chamfer_normals_bwd");
    if (rc) return rc;
    PTK_REQUIRE(grad_cham_normals, PTK_ERR_SHAPE, "chamfer_normals_bwd: null grad_cham_normals pointer");
    if (!grad_xn && !grad_yn) return PTK_OK;
    return pair_bwd<normal_parts>(x_normals, y_normals, len_x, len_y, idx_x, idx_y, grad_cham_normals, B, P1, P2,
                                 reduction == PTK_REDUCE_MEAN ? 1 : 0, grad_xn, grad_yn, as_stream(stream));
}

extern "C" int ptk_chamfer_normals_bwd_det(const float *x_normals, const float *y_normals, const int64_t *len_x,
                                           const int64_t *len_y, const int32_t *idx_x, const int32_t *idx_y,
                                           const float *grad_cham_normals, int64_t B, int64_t P1, int64_t P2,
                                           int reduction, float *grad_xn, float *grad_yn, void *workspace,
                                           size_t workspace_bytes, ptk_stream_t stream) {
    PTK_NVTX("ptk_chamfer_normals_bwd_det");
    int rc = normals_check(x_normals, y_normals, idx_x, idx_y, B, P1, P2, reduction, "chamfer_normals_bwd_det");
    if (rc) return rc;
    PTK_REQUIRE(grad_cham_normals, PTK_ERR_SHAPE, "chamfer_normals_bwd_det: null grad_cham_normals pointer");
    if (!grad_xn && !grad_yn) return PTK_OK;
    rc = det_check_workspace(workspace, workspace_bytes, ptk_chamfer_bwd_det_workspace_bytes(B, P1, P2),
                             "chamfer_normals_bwd_det");
    if (rc) return rc;
    return pair_bwd_det<normal_parts>(x_normals, y_normals, len_x, len_y, idx_x, idx_y, grad_cham_normals, B, P1, P2,
                                     reduction == PTK_REDUCE_MEAN ? 1 : 0, grad_xn, grad_yn, workspace, as_stream(stream));
}
