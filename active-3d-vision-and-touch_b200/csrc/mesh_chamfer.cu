// utils.chamfer_distance(verts, faces, gt_points, num, repeat) on device pointers, one ABI call per pass.
//
// Replaces the body of pterotactyl/utility/utils.py:204-217 -- `repeat` independent samplings of the predicted mesh
// (batch_sample, utils.py:152-187), PyTorch3D's chamfer_distance against the ground-truth cloud for each, the stack and
// the mean -- and its autograd: forward = repeat x (ptk_sample_fwd -> ptk_chamfer_fwd) + the mean, backward = repeat x
// (ptk_chamfer_bwd -> ptk_sample_bwd) accumulated into one vertex gradient (and, for the autoencoder, one gradient of
// the second cloud, autoencoder/train.py:145-150).  The kernels are the ones behind the separate entry points (same
// results); what goes away is the host frame between them: one autograd node instead of 2 x repeat + 2, no
// intermediate torch tensors.  The host-buffer twin is ptk_host_mesh_chamfer (host_api.cu).  ptk_mesh_chamfer_bwd_det
// runs the same loop on the deterministic backward pieces (ptk_chamfer_bwd_det -> ptk_sample_bwd_det).
#include "ptk_common.cuh"

namespace ptk {

// acc = first ? v : acc + v  (the sum of torch.stack(cds)), then the mean's multiply by 1/repeat on the last repeat
__global__ void mc_accumulate_kernel(float *__restrict__ acc, const float *__restrict__ v, long long n, int first,
                                     float final_scale) {
    pdl_wait();
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) {
        const float s = first ? v[i] : acc[i] + v[i];
        acc[i] = final_scale != 1.0f ? s * final_scale : s;
    }
}
__global__ void mc_scale_kernel(float *__restrict__ out, const float *__restrict__ v, float s, long long n) {
    pdl_wait();
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) out[i] = s * v[i];
}

static size_t mc_align(size_t b) { return (b + 255) & ~(size_t)255; }

struct McWs {
    char *sample, *chamfer;
    float *cham, *gc, *gx, *gv, *gy;
    size_t sample_bytes, chamfer_bytes, total;
};
static McWs mc_carve(void *ws, int64_t B, int64_t V, int64_t F, int64_t S, int64_t P2) {
    McWs w;
    size_t off = 0;
    auto take = [&](size_t bytes) { size_t o = off; off += mc_align(bytes); return o; };
    w.sample_bytes = ptk_sample_workspace_bytes(B, F);
    w.chamfer_bytes = ptk_chamfer_workspace_bytes(B, S, P2);
    const size_t o_s = take(w.sample_bytes), o_c = take(w.chamfer_bytes), o_cham = take((size_t)B * 4), o_gc = take((size_t)B * 4);
    const size_t o_gx = take((size_t)B * S * 12), o_gv = take((size_t)B * V * 12), o_gy = take((size_t)B * P2 * 12);
    char *base = reinterpret_cast<char *>(ws);
    w.sample = base + o_s; w.chamfer = base + o_c;
    w.cham = reinterpret_cast<float *>(base + o_cham); w.gc = reinterpret_cast<float *>(base + o_gc);
    w.gx = reinterpret_cast<float *>(base + o_gx); w.gv = reinterpret_cast<float *>(base + o_gv);
    w.gy = reinterpret_cast<float *>(base + o_gy);
    w.total = off;
    return w;
}

}  // namespace ptk

using namespace ptk;

extern "C" size_t ptk_mesh_chamfer_workspace_bytes(int64_t B, int64_t V, int64_t F, int64_t S, int64_t P2) {
    if (B <= 0 || V <= 0 || F <= 0 || S <= 0 || P2 <= 0) return 0;
    return mc_carve(nullptr, B, V, F, S, P2).total;
}

extern "C" int ptk_mesh_chamfer_fwd(const float *verts, int64_t B, int64_t V, const int32_t *faces, int64_t F,
                                    const float *gt, int64_t P2, const float *u_face, const float *uv, int64_t S,
                                    int64_t repeat, float *cd, float *pts, int32_t *face_idx, int32_t *idx_x,
                                    int32_t *idx_y, void *workspace, size_t workspace_bytes, ptk_stream_t stream) {
    PTK_NVTX("ptk_mesh_chamfer_fwd");
    PTK_REQUIRE(verts && faces && gt && uv && cd && pts && face_idx && idx_x && idx_y, PTK_ERR_SHAPE,
                "mesh_chamfer_fwd: null pointer");
    PTK_REQUIRE(B > 0 && V > 0 && F > 0 && P2 > 0 && S > 0 && repeat > 0, PTK_ERR_SHAPE, "mesh_chamfer_fwd: empty input");
    PTK_REQUIRE(workspace && workspace_bytes >= ptk_mesh_chamfer_workspace_bytes(B, V, F, S, P2), PTK_ERR_WORKSPACE,
                "mesh_chamfer_fwd: workspace too small");
    PTK_REQUIRE((reinterpret_cast<uintptr_t>(workspace) & 255) == 0, PTK_ERR_ALIGN, "mesh_chamfer_fwd: workspace must be 256-byte aligned");
    const McWs w = mc_carve(workspace, B, V, F, S, P2);
    cudaStream_t st = as_stream(stream);
    const size_t ns = (size_t)B * S, ny = (size_t)B * P2;
    for (int64_t r = 0; r < repeat; ++r) {
        int rc = ptk_sample_fwd(verts, B, V, faces, F, u_face ? u_face + r * ns : nullptr, uv + r * 2 * ns, S,
                                pts + r * ns * 3, face_idx + r * ns, w.sample, w.sample_bytes, stream);
        if (rc) return rc;
        rc = ptk_chamfer_fwd(pts + r * ns * 3, gt, B, S, P2, nullptr, idx_x + r * ns, nullptr, idx_y + r * ny, w.cham,
                             w.chamfer, w.chamfer_bytes, stream);
        if (rc) return rc;
        // torch.stack(cds).mean(dim=0): the sum in repeat order, then one multiply by 1/repeat
        launch_pdl(mc_accumulate_kernel, dim3((unsigned)ceil_div(B, 256)), dim3(256), 0, st, cd, (const float *)w.cham,
                   (long long)B, r == 0 ? 1 : 0, r == repeat - 1 ? 1.0f / (float)repeat : 1.0f);
        PTK_CHECK_LAUNCH();
    }
    return PTK_OK;
}

// det: the deterministic pieces (ptk_chamfer_bwd_det, ptk_sample_bwd_det), whose workspaces follow the default layout
static int mesh_chamfer_bwd(const float *gt, const float *pts, const int32_t *face_idx, const int32_t *idx_x,
                            const int32_t *idx_y, const float *uv, const int32_t *faces, const float *grad_cd, int64_t B,
                            int64_t V, int64_t F, int64_t S, int64_t P2, int64_t repeat, float *grad_verts, float *grad_gt,
                            void *workspace, size_t workspace_bytes, bool det, ptk_stream_t stream) {
    const char *name = det ? "mesh_chamfer_bwd_det" : "mesh_chamfer_bwd";
    PTK_REQUIRE(gt && pts && face_idx && idx_x && idx_y && uv && faces && grad_cd, PTK_ERR_SHAPE, "%s: null pointer", name);
    PTK_REQUIRE(B > 0 && V > 0 && F > 0 && P2 > 0 && S > 0 && repeat > 0, PTK_ERR_SHAPE, "%s: empty input", name);
    if (!grad_verts && !grad_gt) return PTK_OK;
    const size_t need = det ? ptk_mesh_chamfer_bwd_det_workspace_bytes(B, V, F, S, P2) : ptk_mesh_chamfer_workspace_bytes(B, V, F, S, P2);
    PTK_REQUIRE(workspace && workspace_bytes >= need, PTK_ERR_WORKSPACE, "%s: workspace too small", name);
    PTK_REQUIRE((reinterpret_cast<uintptr_t>(workspace) & 255) == 0, PTK_ERR_ALIGN, "%s: workspace must be 256-byte aligned", name);
    const McWs w = mc_carve(workspace, B, V, F, S, P2);
    char *det_c = reinterpret_cast<char *>(workspace) + w.total;
    const size_t det_c_bytes = ptk_chamfer_bwd_det_workspace_bytes(B, S, P2);
    char *det_s = det_c + mc_align(det_c_bytes);
    const size_t det_s_bytes = ptk_sample_bwd_det_workspace_bytes(B, V);
    cudaStream_t st = as_stream(stream);
    const size_t ns = (size_t)B * S, ny = (size_t)B * P2;
    const long long nv = (long long)B * V * 3, ng = (long long)ny * 3;
    // d mean / d cd_r = 1 / repeat
    launch_pdl(mc_scale_kernel, dim3((unsigned)ceil_div(B, 256)), dim3(256), 0, st, w.gc, grad_cd, 1.0f / (float)repeat, (long long)B);
    PTK_CHECK_LAUNCH();
    for (int64_t r = 0; r < repeat; ++r) {
        float *gy_dst = grad_gt ? (r == 0 ? grad_gt : w.gy) : nullptr;
        float *gx_dst = grad_verts ? w.gx : nullptr;
        int rc = det ? ptk_chamfer_bwd_det(pts + r * ns * 3, gt, nullptr, nullptr, idx_x + r * ns, idx_y + r * ny, w.gc, B, S,
                                           P2, PTK_REDUCE_MEAN, gx_dst, gy_dst, det_c, det_c_bytes, stream)
                     : ptk_chamfer_bwd(pts + r * ns * 3, gt, idx_x + r * ns, idx_y + r * ny, w.gc, B, S, P2, gx_dst, gy_dst,
                                       stream);
        if (rc) return rc;
        if (grad_gt && r > 0) {
            launch_pdl(mc_accumulate_kernel, dim3((unsigned)ceil_div(ng, 256)), dim3(256), 0, st, grad_gt, (const float *)w.gy, ng, 0, 1.0f);
            PTK_CHECK_LAUNCH();
        }
        if (grad_verts) {
            float *gv_dst = r == 0 ? grad_verts : w.gv;
            rc = det ? ptk_sample_bwd_det(w.gx, face_idx + r * ns, uv + r * 2 * ns, faces, B, V, F, S, gv_dst, det_s, det_s_bytes,
                                          stream)
                     : ptk_sample_bwd(w.gx, face_idx + r * ns, uv + r * 2 * ns, faces, B, V, F, S, gv_dst, stream);
            if (rc) return rc;
            if (r > 0) {
                launch_pdl(mc_accumulate_kernel, dim3((unsigned)ceil_div(nv, 256)), dim3(256), 0, st, grad_verts, (const float *)w.gv, nv, 0, 1.0f);
                PTK_CHECK_LAUNCH();
            }
        }
    }
    return PTK_OK;
}

extern "C" int ptk_mesh_chamfer_bwd(const float *gt, const float *pts, const int32_t *face_idx, const int32_t *idx_x,
                                    const int32_t *idx_y, const float *uv, const int32_t *faces, const float *grad_cd,
                                    int64_t B, int64_t V, int64_t F, int64_t S, int64_t P2, int64_t repeat,
                                    float *grad_verts, float *grad_gt, void *workspace, size_t workspace_bytes,
                                    ptk_stream_t stream) {
    PTK_NVTX("ptk_mesh_chamfer_bwd");
    return mesh_chamfer_bwd(gt, pts, face_idx, idx_x, idx_y, uv, faces, grad_cd, B, V, F, S, P2, repeat, grad_verts, grad_gt,
                            workspace, workspace_bytes, false, stream);
}

// the default workspace followed by those of ptk_chamfer_bwd_det (B, S, P2) and ptk_sample_bwd_det (B, V)
extern "C" size_t ptk_mesh_chamfer_bwd_det_workspace_bytes(int64_t B, int64_t V, int64_t F, int64_t S, int64_t P2) {
    if (B <= 0 || V <= 0 || F <= 0 || S <= 0 || P2 <= 0) return 0;
    return mc_carve(nullptr, B, V, F, S, P2).total + mc_align(ptk_chamfer_bwd_det_workspace_bytes(B, S, P2)) +
           mc_align(ptk_sample_bwd_det_workspace_bytes(B, V));
}

extern "C" int ptk_mesh_chamfer_bwd_det(const float *gt, const float *pts, const int32_t *face_idx, const int32_t *idx_x,
                                        const int32_t *idx_y, const float *uv, const int32_t *faces, const float *grad_cd,
                                        int64_t B, int64_t V, int64_t F, int64_t S, int64_t P2, int64_t repeat,
                                        float *grad_verts, float *grad_gt, void *workspace, size_t workspace_bytes,
                                        ptk_stream_t stream) {
    PTK_NVTX("ptk_mesh_chamfer_bwd_det");
    return mesh_chamfer_bwd(gt, pts, face_idx, idx_x, idx_y, uv, faces, grad_cd, B, V, F, S, P2, repeat, grad_verts, grad_gt,
                            workspace, workspace_bytes, true, stream);
}
