// Backward of a per-query loss on the two directions of a cloud pair: the Chamfer distance (chamfer.cu) and the Chamfer
// normal term (chamfer_normals.cu).  Thread i of grid (ceil(max(P1,P2) / 256), B) owns x-query i (against y) and
// y-query i (against x).  A valid query's term has an "own" part on its own row and a "near" part on the row of its
// nearest neighbour j in the other cloud.  A PairParts function states the per-query arithmetic
// (qb / tb: the query and target arrays of the pair, idx: the query direction's indices, g: the pair's upstream
// gradient; false: no parts).
//   default: own parts as plain stores (every row of a requested gradient written, 0 without a part), then near parts
//            with fp32 atomics;
//   det:     the scheme of det_accum.cuh.  M_b and the scatter into one cloud take the parts of both directions, so each
//            gradient has the same bits whether or not the other one is requested; a row receives its own part and at
//            most l_other near parts, n = max(lx, ly) + 1.
#pragma once
#include "det_accum.cuh"

namespace ptk {

constexpr int PB_THREADS = 256;

typedef bool (*PairParts)(const float *qb, const float *tb, const int32_t *idx, float g, int i, int Lq, int Lt, int mean,
                          int &j, float own[3], float near[3]);

template <PairParts parts>
__global__ void __launch_bounds__(PB_THREADS)
pair_bwd_own_kernel(const float *__restrict__ x, const float *__restrict__ y, const int32_t *__restrict__ idx_x,
                    const int32_t *__restrict__ idx_y, const float *__restrict__ grad, int P1, int P2,
                    const int64_t *__restrict__ len_x, const int64_t *__restrict__ len_y, int mean,
                    float *__restrict__ grad_x, float *__restrict__ grad_y) {
    pdl_wait();  // launched with programmatic stream serialization (ptk_common.cuh)
    const int b = blockIdx.y;
    const int i = blockIdx.x * PB_THREADS + threadIdx.x;
    const float g = grad[b];
    const float *xb = x + (size_t)b * P1 * 3, *yb = y + (size_t)b * P2 * 3;
    const int L1 = pair_len(len_x, b, P1), L2 = pair_len(len_y, b, P2);
    float own[3], near[3];
    int j;
    if (grad_x && i < P1) {
        float *o = grad_x + ((size_t)b * P1 + i) * 3;
        const bool t = parts(xb, yb, idx_x + (size_t)b * P1, g, i, L1, L2, mean, j, own, near);
        o[0] = t ? own[0] : 0.0f;
        o[1] = t ? own[1] : 0.0f;
        o[2] = t ? own[2] : 0.0f;
    }
    if (grad_y && i < P2) {
        float *o = grad_y + ((size_t)b * P2 + i) * 3;
        const bool t = parts(yb, xb, idx_y + (size_t)b * P2, g, i, L2, L1, mean, j, own, near);
        o[0] = t ? own[0] : 0.0f;
        o[1] = t ? own[1] : 0.0f;
        o[2] = t ? own[2] : 0.0f;
    }
}

// x-queries' near parts into grad_y, y-queries' into grad_x (RED.ADD.F32)
template <PairParts parts>
__global__ void __launch_bounds__(PB_THREADS)
pair_bwd_near_kernel(const float *__restrict__ x, const float *__restrict__ y, const int32_t *__restrict__ idx_x,
                     const int32_t *__restrict__ idx_y, const float *__restrict__ grad, int P1, int P2,
                     const int64_t *__restrict__ len_x, const int64_t *__restrict__ len_y, int mean,
                     float *__restrict__ grad_x, float *__restrict__ grad_y) {
    pdl_wait();
    const int b = blockIdx.y;
    const int i = blockIdx.x * PB_THREADS + threadIdx.x;
    const float g = grad[b];
    const float *xb = x + (size_t)b * P1 * 3, *yb = y + (size_t)b * P2 * 3;
    const int L1 = pair_len(len_x, b, P1), L2 = pair_len(len_y, b, P2);
    float own[3], near[3];
    int j;
    if (grad_y && parts(xb, yb, idx_x + (size_t)b * P1, g, i, L1, L2, mean, j, own, near)) {
        float *o = grad_y + ((size_t)b * P2 + j) * 3;
        atomicAdd(o + 0, near[0]);
        atomicAdd(o + 1, near[1]);
        atomicAdd(o + 2, near[2]);
    }
    if (grad_x && parts(yb, xb, idx_y + (size_t)b * P2, g, i, L2, L1, mean, j, own, near)) {
        float *o = grad_x + ((size_t)b * P1 + j) * 3;
        atomicAdd(o + 0, near[0]);
        atomicAdd(o + 1, near[1]);
        atomicAdd(o + 2, near[2]);
    }
}

// det phase 1: M_b over both directions' parts; the rows of the requested gradients zeroed
template <PairParts parts>
__global__ void __launch_bounds__(PB_THREADS)
pair_bwd_det_max_kernel(const float *__restrict__ x, const float *__restrict__ y, const int32_t *__restrict__ idx_x,
                        const int32_t *__restrict__ idx_y, const float *__restrict__ grad, int P1, int P2,
                        const int64_t *__restrict__ len_x, const int64_t *__restrict__ len_y, int mean,
                        float *__restrict__ grad_x, float *__restrict__ grad_y, unsigned long long *__restrict__ acc_x,
                        unsigned long long *__restrict__ acc_y, unsigned int *__restrict__ mbits) {
    pdl_wait();
    const int b = blockIdx.y;
    const int i = blockIdx.x * PB_THREADS + threadIdx.x;
    const float g = grad[b];
    const float *xb = x + (size_t)b * P1 * 3, *yb = y + (size_t)b * P2 * 3;
    const int L1 = pair_len(len_x, b, P1), L2 = pair_len(len_y, b, P2);
    float m = 0.0f, own[3], near[3];
    int j;
    if (parts(xb, yb, idx_x + (size_t)b * P1, g, i, L1, L2, mean, j, own, near))
#pragma unroll
        for (int d = 0; d < 3; ++d) m = fmaxf(m, fmaxf(det_abs_finite(own[d]), det_abs_finite(near[d])));
    if (parts(yb, xb, idx_y + (size_t)b * P2, g, i, L2, L1, mean, j, own, near))
#pragma unroll
        for (int d = 0; d < 3; ++d) m = fmaxf(m, fmaxf(det_abs_finite(own[d]), det_abs_finite(near[d])));
    if (grad_x && i < P1) det_zero_row(acc_x, grad_x, (size_t)b * P1 + i);
    if (grad_y && i < P2) det_zero_row(acc_y, grad_y, (size_t)b * P2 + i);
    det_block_max<PB_THREADS>(m, mbits + b);
}

// det phase 2: both parts of x-query i and of y-query i
template <PairParts parts>
__global__ void __launch_bounds__(PB_THREADS)
pair_bwd_det_add_kernel(const float *__restrict__ x, const float *__restrict__ y, const int32_t *__restrict__ idx_x,
                        const int32_t *__restrict__ idx_y, const float *__restrict__ grad, int P1, int P2,
                        const int64_t *__restrict__ len_x, const int64_t *__restrict__ len_y, int mean,
                        float *__restrict__ grad_x, float *__restrict__ grad_y, unsigned long long *__restrict__ acc_x,
                        unsigned long long *__restrict__ acc_y, const unsigned int *__restrict__ mbits, DetBound nb) {
    pdl_wait();
    const int b = blockIdx.y;
    const int i = blockIdx.x * PB_THREADS + threadIdx.x;
    const float g = grad[b];
    const float *xb = x + (size_t)b * P1 * 3, *yb = y + (size_t)b * P2 * 3;
    const int L1 = pair_len(len_x, b, P1), L2 = pair_len(len_y, b, P2);
    const double scale = det_scale(mbits, nb, b);
    const size_t bx = (size_t)b * P1 * 3, by = (size_t)b * P2 * 3;
    float own[3], near[3];
    int j;
    if (parts(xb, yb, idx_x + (size_t)b * P1, g, i, L1, L2, mean, j, own, near))
#pragma unroll
        for (int d = 0; d < 3; ++d) {
            if (grad_x) det_add(acc_x + bx + (size_t)i * 3 + d, grad_x + bx + (size_t)i * 3 + d, own[d], scale);
            if (grad_y) det_add(acc_y + by + (size_t)j * 3 + d, grad_y + by + (size_t)j * 3 + d, near[d], scale);
        }
    if (parts(yb, xb, idx_y + (size_t)b * P2, g, i, L2, L1, mean, j, own, near))
#pragma unroll
        for (int d = 0; d < 3; ++d) {
            if (grad_y) det_add(acc_y + by + (size_t)i * 3 + d, grad_y + by + (size_t)i * 3 + d, own[d], scale);
            if (grad_x) det_add(acc_x + bx + (size_t)j * 3 + d, grad_x + bx + (size_t)j * 3 + d, near[d], scale);
        }
}

// the default pair; the caller has checked its arguments and that a gradient is requested
template <PairParts parts>
int pair_bwd(const float *x, const float *y, const int64_t *len_x, const int64_t *len_y, const int32_t *idx_x,
             const int32_t *idx_y, const float *grad, int64_t B, int64_t P1, int64_t P2, int mean, float *grad_x,
             float *grad_y, cudaStream_t st) {
    const dim3 grid((unsigned)ceil_div(P1 > P2 ? P1 : P2, PB_THREADS), (unsigned)B);
    launch_pdl(pair_bwd_own_kernel<parts>, grid, dim3(PB_THREADS), 0, st, x, y, idx_x, idx_y, grad, (int)P1, (int)P2,
               len_x, len_y, mean, grad_x, grad_y);
    PTK_CHECK_LAUNCH();
    launch_pdl(pair_bwd_near_kernel<parts>, grid, dim3(PB_THREADS), 0, st, x, y, idx_x, idx_y, grad, (int)P1, (int)P2,
               len_x, len_y, mean, grad_x, grad_y);
    PTK_CHECK_LAUNCH();
    return PTK_OK;
}

// the det triple on a det_workspace_bytes(B, P1, P2) workspace (checked by the caller)
template <PairParts parts>
int pair_bwd_det(const float *x, const float *y, const int64_t *len_x, const int64_t *len_y, const int32_t *idx_x,
                 const int32_t *idx_y, const float *grad, int64_t B, int64_t P1, int64_t P2, int mean, float *grad_x,
                 float *grad_y, void *workspace, cudaStream_t st) {
    DetWs w;
    PTK_CHECK_CUDA(det_begin(workspace, B, P1, st, w));
    const DetBound nb = det_bound_len(len_x, P1, len_y, P2);
    const dim3 grid((unsigned)ceil_div(P1 > P2 ? P1 : P2, PB_THREADS), (unsigned)B);
    launch_pdl(pair_bwd_det_max_kernel<parts>, grid, dim3(PB_THREADS), 0, st, x, y, idx_x, idx_y, grad, (int)P1, (int)P2,
               len_x, len_y, mean, grad_x, grad_y, w.acc_a, w.acc_b, w.mbits);
    PTK_CHECK_LAUNCH();
    launch_pdl(pair_bwd_det_add_kernel<parts>, grid, dim3(PB_THREADS), 0, st, x, y, idx_x, idx_y, grad, (int)P1, (int)P2,
               len_x, len_y, mean, grad_x, grad_y, w.acc_a, w.acc_b, (const unsigned int *)w.mbits, nb);
    PTK_CHECK_LAUNCH();
    det_launch_convert<PB_THREADS>(w, nb, B, grad_x, P1, grad_y, P2, st);
    PTK_CHECK_LAUNCH();
    return PTK_OK;
}

}  // namespace ptk
