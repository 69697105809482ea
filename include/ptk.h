/*
 * ptk.h -- C ABI of libptk_b200.so: the B200 (sm_100a) reconstruction hot path of pterotactyl.
 *
 * This is the drop-in boundary (SURVEY.md 8b).  The reference has no FFI of its own: the hot path
 * is reached through Python signatures that bottom out in PyTorch3D's `_C` extension and ATen.
 * Each entry point below names the reference call (file:line under /root/reference, or the
 * un-vendored PyTorch3D 0.5.0 symbol) it replaces.  INTEGRATION.md shows the ctypes binding a
 * maintainer of the reference would add.
 *
 * Conventions
 *   - plain C: pointers + sizes, no torch types.  Unless a parameter is documented as HOST, every
 *     pointer is a DEVICE pointer on the current CUDA device, owned by the caller; the library never
 *     allocates or frees caller-visible memory (workspaces are passed in).
 *   - every call is asynchronous on `stream` (a cudaStream_t passed as void*), performs no host
 *     synchronisation and is safe under CUDA-graph capture.  The ptk_host_* family is the exception:
 *     it takes HOST buffers, copies both ways and synchronises its own stream.
 *   - return value: 0 (PTK_OK) or a negative PTK_ERR_*; ptk_last_error() gives a thread-local
 *     message.  The reference raises ValueError on shape mismatch (PyTorch3D) -- the Python host
 *     layer maps PTK_ERR_SHAPE to ValueError and the rest to RuntimeError.
 *   - all float tensors are fp32, C-contiguous; indices are int32 at this ABI (int64 at the torch
 *     boundary, converted by the host layer).
 */
#ifndef PTK_H_
#define PTK_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define PTK_ABI_VERSION 1

#define PTK_OK 0
#define PTK_ERR_SHAPE (-1)     /* bad sizes / null pointer where one is required */
#define PTK_ERR_ALIGN (-2)     /* pointer not aligned as documented */
#define PTK_ERR_ARCH (-3)      /* device is not sm_100 */
#define PTK_ERR_CUDA (-4)      /* a CUDA runtime call failed (message has the cudaError string) */
#define PTK_ERR_WORKSPACE (-5) /* workspace too small */

typedef void *ptk_stream_t; /* cudaStream_t */

int ptk_version(void);
const char *ptk_last_error(void);
/* SM count, max SM clock (kHz), L2 bytes, opt-in shared memory per block, compute capability. */
int ptk_device_info(int device, int *sm_count, int *clock_khz, int *l2_bytes, int *smem_optin,
                    int *cc_major, int *cc_minor);
/* Number of kernels this library has launched in the calling process so far (all threads, all streams; launches
 * recorded into a CUDA graph count once, at capture).  No reference counterpart: it lets a harness state how many of
 * the library's own kernels ran inside a timed region (bench.py `gpu_launches`) instead of assuming it. */
uint64_t ptk_launch_count(void);

/* ------------------------------------------------------------------------------------------------
 * Chamfer distance / 1-NN between point clouds.
 * Replaces pytorch3d.loss.chamfer_distance(x, y, batch_reduction=None) and pytorch3d.ops.knn_points
 * (K=1) -- PyTorch3D 0.5.0 `_C.knn_points_idx` / `_C.knn_points_backward` -- as called from
 * pterotactyl/utility/utils.py:207,212.
 *   x (B,P1,3), y (B,P2,3).  Squared L2, dist = fma(dz,dz, fma(dy,dy, dx*dx)) (the arithmetic
 *   PyTorch3D's CUDA kernel executes), strict '<' scanning targets in ascending order: the lowest
 *   index wins exact ties.  cham[b] = mean_i dist_x[b,i] + mean_j dist_y[b,j].
 * ---------------------------------------------------------------------------------------------- */
size_t ptk_chamfer_workspace_bytes(int64_t B, int64_t P1, int64_t P2); /* 16-byte aligned workspace */

/* Nearest-neighbour scan algorithm (process-wide; all give bit-identical results):
 *   PTK_CHAMFER_FILTER            3-FFMA expansion filter on packed FP32x2 + exact recheck/rescue
 *   PTK_CHAMFER_EXACT             the defining 6-op arithmetic for every (query, target) pair
 *   PTK_CHAMFER_PRUNED            cell-sorted clouds + box hierarchy: only the leaves whose lower bound can beat or
 *                                 tie a query's incumbent are evaluated (same arithmetic, same tie rule); clouds of
 *                                 more than 524288 points fall back to PTK_CHAMFER_FILTER
 *   PTK_CHAMFER_AUTO (default)    PTK_CHAMFER_PRUNED when both clouds have >= PTK_CHAMFER_AUTO_MIN_POINTS points,
 *                                 PTK_CHAMFER_FILTER otherwise */
#define PTK_CHAMFER_FILTER 0
#define PTK_CHAMFER_EXACT 1
#define PTK_CHAMFER_PRUNED 2
#define PTK_CHAMFER_AUTO 3
#define PTK_CHAMFER_AUTO_MIN_POINTS 20000
int ptk_chamfer_set_algo(int algo);
int ptk_chamfer_get_algo(void);
/* Diagnostics (synchronises `stream`): number of queries of the last forward that used `workspace`
 * whose filter result was ambiguous and went through the exact rescue scan. */
int ptk_chamfer_rescued(const void *workspace, int64_t B, int64_t P1, int64_t P2, int64_t *n_rescued,
                        ptk_stream_t stream);

/* One direction: for every p1[b,i] its nearest p2[b,j].  dist (B,P1) and/or idx (B,P1) may be NULL. */
int ptk_knn1_fwd(const float *p1, const float *p2, int64_t B, int64_t P1, int64_t P2, float *dist,
                 int32_t *idx, void *workspace, size_t workspace_bytes, ptk_stream_t stream);

/* Both directions in one launch + fused mean reduction.  dist_x/dist_y may be NULL; idx_x (B,P1),
 * idx_y (B,P2) and cham (B) are required (idx feeds the backward). */
int ptk_chamfer_fwd(const float *x, const float *y, int64_t B, int64_t P1, int64_t P2, float *dist_x,
                    int32_t *idx_x, float *dist_y, int32_t *idx_y, float *cham, void *workspace,
                    size_t workspace_bytes, ptk_stream_t stream);

/* Gradient of cham w.r.t. x and y (either may be NULL: the autoencoder only needs grad_y,
 * pterotactyl/reconstruction/autoencoder/train.py:145-151).  grad_* are fully overwritten. */
int ptk_chamfer_bwd(const float *x, const float *y, const int32_t *idx_x, const int32_t *idx_y,
                    const float *grad_cham, int64_t B, int64_t P1, int64_t P2, float *grad_x,
                    float *grad_y, ptk_stream_t stream);

/* Ragged batches: clouds of different sizes padded to (B,P1,3) / (B,P2,3), as PyTorch3D batches them.
 *   len_x / len_y (resp. len1 / len2) are DEVICE int64 arrays of B lengths; NULL means every cloud is full.  Each
 *   value is clamped to [0, P] on the device; the host never reads them, so a call needs no synchronisation and can
 *   be captured in a CUDA graph with the lengths changed in place between replays.  For pair b only x[b, :lx] and
 *   y[b, :ly] exist: padding is never read into a result, whatever it holds.
 *   - valid queries: dist / idx bit-identical to a homogeneous call on the sliced pair (same arithmetic, same
 *     lowest-index tie rule), and so is cham[b];
 *   - padded queries (i >= len) and valid queries whose target cloud is empty: dist = 0, idx = 0 (PyTorch3D's zero
 *     fill);
 *   - reduction PTK_REDUCE_MEAN: cham[b] = sum_x / max(lx, 1) + sum_y / max(ly, 1).  An empty cloud contributes 0
 *     (the divisor is clamped to 1, as current PyTorch3D releases clamp their lengths; 0.5.0's behaviour for a zero
 *     length is not pinned here).  PTK_REDUCE_SUM: cham[b] = sum_x + sum_y.  Any other value is PTK_ERR_SHAPE;
 *   - backward: the valid points of pair b get the gradient of its own term (scale 1 / max(len, 1) for mean, 1 for
 *     sum); padded points get exactly 0 and queries with an empty target cloud contribute nothing.  grad_* are
 *     fully overwritten.
 * The workspace is ptk_chamfer_workspace_bytes(B, P1, P2) and ptk_chamfer_rescued works after these calls.  The
 * homogeneous entry points above are these calls with NULL lengths and PTK_REDUCE_MEAN.
 * Replace pytorch3d.loss.chamfer_distance(x, y, x_lengths, y_lengths, point_reduction=...) and
 * pytorch3d.ops.knn_points(p1, p2, lengths1, lengths2, K=1) of PyTorch3D 0.5.0. */
#define PTK_REDUCE_MEAN 0
#define PTK_REDUCE_SUM 1
int ptk_chamfer_fwd_lengths(const float *x, const float *y, const int64_t *len_x, const int64_t *len_y, int64_t B,
                            int64_t P1, int64_t P2, int reduction, float *dist_x, int32_t *idx_x, float *dist_y,
                            int32_t *idx_y, float *cham, void *workspace, size_t workspace_bytes, ptk_stream_t stream);
int ptk_chamfer_bwd_lengths(const float *x, const float *y, const int64_t *len_x, const int64_t *len_y,
                            const int32_t *idx_x, const int32_t *idx_y, const float *grad_cham, int64_t B, int64_t P1,
                            int64_t P2, int reduction, float *grad_x, float *grad_y, ptk_stream_t stream);
int ptk_knn1_fwd_lengths(const float *p1, const float *p2, const int64_t *len1, const int64_t *len2, int64_t B,
                         int64_t P1, int64_t P2, float *dist, int32_t *idx, void *workspace, size_t workspace_bytes,
                         ptk_stream_t stream);

/* ------------------------------------------------------------------------------------------------
 * Area-weighted surface sampling.  Replaces the body of utils.batch_sample
 * (pterotactyl/utility/utils.py:152-187): pytorch3d mesh_face_areas_normals (utils.py:164), the NaN
 * guards (165-168), Tensor.multinomial (170), _rand_barycentric_coords (179) and the barycentric
 * interpolation (182-185), fused.
 *   verts (B,V,3); faces (F,3) int32 shared by the batch; u_face (B,S) and uv (2,B,S) are the
 *   uniform [0,1) draws (the RNG stream); pts (B,S,3); face_idx (B,S) int32 (saved for backward).
 * Face choice uses an order-independent integer prefix sum (see oracle/ptk_oracle.c) so the result
 * is bit-exact for a given uniform stream.
 * u_face may be NULL: face_idx (B,S) is then an INPUT -- the faces were drawn by the caller (the host
 * layer's face_draw="multinomial" mode lets ATen's own Tensor.multinomial draw them, which reproduces
 * the reference's RNG stream) -- and only the interpolation runs; workspace is not used.
 * ---------------------------------------------------------------------------------------------- */
size_t ptk_sample_workspace_bytes(int64_t B, int64_t F);
int ptk_sample_fwd(const float *verts, int64_t B, int64_t V, const int32_t *faces, int64_t F,
                   const float *u_face, const float *uv, int64_t S, float *pts, int32_t *face_idx,
                   void *workspace, size_t workspace_bytes, ptk_stream_t stream);
/* grad_verts (B,V,3) is fully overwritten:  grad_verts[b, faces[f,k]] += w_k * grad_pts[b,s]. */
int ptk_sample_bwd(const float *grad_pts, const int32_t *face_idx, const float *uv,
                   const int32_t *faces, int64_t B, int64_t V, int64_t F, int64_t S,
                   float *grad_verts, ptk_stream_t stream);

/* Face areas of a batch of meshes sharing one face list: verts (B,V,3), faces (F,3) int32 -> areas (B,F); what
 * utils.batch_sample computes at utils.py:163-164 before normalising (NaN areas are left for the caller's guards). */
int ptk_mesh_face_areas(const float *verts, int64_t B, int64_t V, const int32_t *faces, int64_t F, float *areas,
                        ptk_stream_t stream);

/* pytorch3d.ops.mesh_face_areas_normals(verts, faces) drop-in (utils.py:21,164): packed verts (V,3),
 * int64 faces (F,3) -> areas (F), unit normals (F,3) (normals may be NULL). */
int ptk_face_areas_normals(const float *verts, int64_t V, const int64_t *faces, int64_t F, float *areas,
                           float *normals, ptk_stream_t stream);

/* ------------------------------------------------------------------------------------------------
 * GCN vertex aggregation.  Replaces the dense `torch.matmul(adj, features[:, :, :length])` + concat +
 * bias + activation of GCN_layer.forward (pterotactyl/reconstruction/vision/model.py:354-363, copies
 * at autoencoder/model.py:112-124 and policies/DDQN/model.py:148-160) with a CSR gather.
 *   out[b,i,c] = act( sum_e val[e] * in[b,col[e],c] + bias[c] )   for c <  L, e in row i
 *   out[b,i,c] = act( in[b,i,c] )                                  for c >= L
 * in/out (B,Nv,C) with C % 4 == 0 and 16-byte aligned bases for the vector path (any C works,
 * scalar path otherwise).  bias may be NULL.  hubs (n_hubs int32 row ids, may be NULL) lists the
 * rows of degree > 128 (touch-chart centre vertices, utils.py:95-98): each is processed by a whole
 * CTA instead of one warp.  The backward w.r.t. `in` is the same call on the
 * transposed graph with bias = NULL, relu = 0 (the activation mask is applied by the producer of
 * the incoming gradient, see ptk_gcn_linear_dgrad).
 * ---------------------------------------------------------------------------------------------- */
int ptk_gcn_aggregate(const int32_t *rowptr, const int32_t *col, const float *val,
                      const int32_t *hubs, int32_t n_hubs, int64_t Nv, const float *in, int64_t B,
                      int64_t C, int64_t L, const float *bias, int relu, float *out,
                      ptk_stream_t stream);
/* Same, with the hub rows factored over a common neighbour set S (ptk_b200/graph.py builds it): for the
 * rows listed in `hubs`
 *     out[b,h,:L] = act( hub_alpha[h] * sum_{k<n_common} common_w[k] * in[b,common_col[k],:L]
 *                        + sum_{e in row h of the (reduced) CSR} val[e] * in[b,col[e],:L] + bias )
 * so the ~1150 boundary rows every touch-chart centre vertex is linked to (utils.py:126-128) are read once
 * per batch element instead of once per hub row.  row_skip (Nv bytes) flags the hub rows.  n_common = 0
 * (all common_* / hub_alpha / row_skip NULL) is exactly ptk_gcn_aggregate.  Needs the vector path
 * (C % 4 == 0, 16-byte aligned, 1 <= L, L <= 384).
 * ldi / ldo: row strides (floats) of in / out, 0 = C.  With ptk_gcn_linear_fwd_split this is the fused
 * layer: in = the compact (B,Nv,n_split) head the GEMM wrote, C = n_split, ldo = layer width. */
int ptk_gcn_aggregate_ex(const int32_t *rowptr, const int32_t *col, const float *val,
                         const int32_t *hubs, int32_t n_hubs, const int32_t *common_col,
                         const float *common_w, int32_t n_common, const float *hub_alpha,
                         const uint8_t *row_skip, int64_t Nv, const float *in, int64_t B, int64_t C,
                         int64_t L, const float *bias, int relu, float *out, int64_t ldi, int64_t ldo,
                         ptk_stream_t stream);
/* ptk_gcn_aggregate_ex with per-tile neighbour unions (csrc/gcn_aggregate_union.cu).  The rows of a tile of 8
 * consecutive vertices share most of their neighbours; the caller lists, per tile, the sorted union of the neighbour
 * columns of its non-hub rows: tile_uptr (ceil(Nv/8)+1 offsets), tile_ucol, and per CSR entry e the index
 * tile_lidx[e] of col[e] in its tile's union; max_union = the largest union.  mode:
 *   PTK_AGG_AUTO        the form measured fastest for the shape (dense tile for > 128 aggregated channels and for
 *                       inputs without pass-through columns; the L2 gather otherwise)
 *   PTK_AGG_L2_GATHER   ptk_gcn_aggregate_ex
 *   PTK_AGG_DENSE_TILE  a warp owns the tile for one batch element: out[8 x C'] = A[8 x U] . X[U x C'], every union row
 *                       read from L2 once and accumulated into up to 8 register rows, A (0 where unused) in shared memory
 *   PTK_AGG_RING        union rows staged in shared memory by cp.async through an mbarrier ring, gathered with LDS
 *                       (measured slower than the L2 gather on B200; kept for comparison)
 * All forms add a row's neighbours in ascending column order: identical results (for finite inputs in the dense form,
 * where an unused column contributes fma(0, x, acc)).  Falls back to ptk_gcn_aggregate_ex when the tile arrays are NULL
 * or the shape is outside the kernels' range (unions above 256 rows, non-vector shapes). */
enum { PTK_AGG_AUTO = 0, PTK_AGG_L2_GATHER = 1, PTK_AGG_DENSE_TILE = 2, PTK_AGG_RING = 3 };
int ptk_gcn_aggregate_tiled(const int32_t *rowptr, const int32_t *col, const float *val, const int32_t *hubs,
                            int32_t n_hubs, const int32_t *common_col, const float *common_w, int32_t n_common,
                            const float *hub_alpha, const uint8_t *row_skip, const int32_t *tile_uptr,
                            const int32_t *tile_ucol, const uint16_t *tile_lidx, int32_t max_union, int32_t mode,
                            int64_t Nv, const float *in, int64_t B, int64_t C, int64_t L, const float *bias, int relu,
                            float *out, int64_t ldi, int64_t ldo, ptk_stream_t stream);
/* gbias[c] = sum_{rows} g[row,c] for c < L, 0 for L <= c < C  (g is (M,C)); overwrites gbias.
 * Deterministic two-stage column sum; workspace from ptk_gcn_bias_grad_workspace_bytes. */
size_t ptk_gcn_bias_grad_workspace_bytes(int64_t M, int64_t L);
int ptk_gcn_bias_grad(const float *g, int64_t M, int64_t C, int64_t L, float *gbias, void *workspace,
                      size_t workspace_bytes, ptk_stream_t stream);
/* The same for n_mats gradient matrices stored back to back (g: n_mats x M x C, gbias: n_mats x C) in two
 * launches: the layers of one GCN backward pass write their output gradients into one slab. */
size_t ptk_gcn_bias_grad_batched_workspace_bytes(int64_t n_mats, int64_t M, int64_t L);
int ptk_gcn_bias_grad_batched(const float *g, int64_t n_mats, int64_t M, int64_t C, int64_t L, float *gbias,
                              void *workspace, size_t workspace_bytes, ptk_stream_t stream);

/* out[i] = act[i] > 0 ? g[i] : 0 -- ReLU backward where it cannot be fused into a dgrad epilogue. */
int ptk_relu_mask(const float *g, const float *act, int64_t n, float *out, ptk_stream_t stream);

/* ------------------------------------------------------------------------------------------------
 * GCN per-vertex linear layer.  Replaces `torch.matmul(features, self.weight)`
 * (vision/model.py:352) and its autograd.
 *   fwd   : H (M,N)  = X (M,K) . W (K,N)
 *   dgrad : gX (M,K) = gH (M,N) . W^T, optionally masked by (act[m,k] > 0) -- the ReLU of the
 *           previous layer (vision/model.py:324) fused into the epilogue; act may be NULL.
 * Where the layer is a true GEMM (reduction >= 32, >= 16 output columns, 16-byte aligned rows) fwd and
 * dgrad run on the tcgen05 tensor cores with the error-compensated 3xTF32 scheme (FP32-level accuracy,
 * csrc/gemm_tf32x3.cu); otherwise on exact-FP32 FFMA kernels (csrc/gcn_linear.cu).
 *   wgrad : gW (K,N) = X^T . gH  (overwrites gW; the sum over the M rows is split across CTAs and
 *           reduced in a fixed order through the workspace => deterministic)
 * ---------------------------------------------------------------------------------------------- */
/* Workspace of fwd and dgrad: the split weights, the packed ReLU mask and one partial output tile + flag per
 * persistent CTA (the tensor-core kernel deals its k-blocks out evenly; a tile shared by two CTAs is combined
 * through that slot in a fixed order).  One workspace must not be shared by calls running concurrently. */
size_t ptk_gcn_linear_workspace_bytes(int64_t M, int64_t K, int64_t N);
/* algo: PTK_GEMM_AUTO (tensor cores where eligible), PTK_GEMM_FFMA (exact-FP32 FFMA, k-sequential
 * accumulation like a scalar FP32 loop) or PTK_GEMM_TF32X3 (error if the shape is not eligible). */
#define PTK_GEMM_AUTO 0
#define PTK_GEMM_FFMA 1
#define PTK_GEMM_TF32X3 2
int ptk_gcn_linear_fwd(const float *X, const float *W, int64_t M, int64_t K, int64_t N, float *H, int algo,
                       void *workspace, size_t workspace_bytes, ptk_stream_t stream);
/* Fused GCN-layer forward GEMM (exact-FP32 kernel): H = X.W is never materialised as one matrix --
 * columns [0, n_split) go to `head` (M, n_split) for ptk_gcn_aggregate_ex, columns [n_split, N) are
 * ReLU'd (relu != 0) and written straight into `out` (M, N): GCN_layer.forward's `cat(adj @ H[:, :L],
 * H[:, L:])` + activation (vision/model.py:355-363) without the round trip of the pass-through slice.
 * n_split = L rounded up to a multiple of 4; needs K % 4 == 0, N % 4 == 0, N >= 64, 16-byte alignment.
 * x_bits (optional, M x ceil(K/32) words, K <= 512): by-product for the backward -- bit (k & 31) of word
 * [m * ceil(K/32) + (k >> 5)] = X[m,k] > 0, the packed ReLU mask ptk_gcn_linear_dgrad takes as act_bits. */
int ptk_gcn_linear_fwd_split(const float *X, const float *W, int64_t M, int64_t K, int64_t N, int64_t n_split,
                             float *head, float *out, int relu, uint32_t *x_bits, ptk_stream_t stream);
/* act (optional, M x K): gX is masked by act > 0 (ReLU backward of the layer input).  act_bits (optional): the
 * same mask already packed by ptk_gcn_linear_fwd_split; without it the tensor-core path packs `act` itself. */
int ptk_gcn_linear_dgrad(const float *gH, const float *W, const float *act, const uint32_t *act_bits, int64_t M,
                         int64_t K, int64_t N, float *gX, int algo, void *workspace, size_t workspace_bytes,
                         ptk_stream_t stream);
size_t ptk_gcn_linear_wgrad_workspace_bytes(int64_t M, int64_t K, int64_t N);
int ptk_gcn_linear_wgrad(const float *X, const float *gH, int64_t M, int64_t K, int64_t N, float *gW,
                         int algo, void *workspace, size_t workspace_bytes, ptk_stream_t stream);

/* ------------------------------------------------------------------------------------------------
 * A whole GCN.forward / its backward in ONE call (pterotactyl/reconstruction/vision/model.py:316-331; the copies in
 * autoencoder/model.py:85-92 and policies/DDQN/model.py:122-127).  Walks the layers in native code with exactly the
 * kernels, order and results of the per-layer entry points above -- what changes is that no host-language frame sits
 * between two launches (the per-layer kernels are 5-135 us at the training batch).
 *
 * ptk_gcn_csr: one direction of the adjacency (A^ for the forward, its transpose for the backward) in both forms the
 * aggregation takes: the plain CSR + hub list (ptk_gcn_aggregate) and the kernel form with the hub rows' common
 * neighbour set split off (ptk_gcn_aggregate_ex; n_common == 0: absent, k_* may then equal the plain arrays).
 *
 * Layer l maps width[l] -> width[l+1] channels, propagates its first Ls[l] output channels through the adjacency and
 * applies ReLU iff relus[l].  W[l] (width[l] x width[l+1]) row-major, bias[l] (width[l+1]); acts[l] (B,Nv,width[l+1])
 * receives the output of layer l (in inference the caller may alternate two buffers).  x_bits (array of n_layers
 * pointers, entries or the array itself may be NULL): x_bits[l] (B*Nv x ceil(width[l]/32) words) receives the packed
 * ReLU mask of layer l's INPUT as a by-product of the fused forward, for this layer's dgrad.  algo: PTK_GEMM_* of the
 * forward GEMMs; fuse != 0 enables the split-epilogue GEMM + strided aggregate for 'cut' ReLU layers (FFMA only).
 * ---------------------------------------------------------------------------------------------- */
typedef struct ptk_gcn_csr {
    const int32_t *rowptr, *col; const float *val; const int32_t *hubs; int32_t n_hubs;
    const int32_t *k_rowptr, *k_col; const float *k_val; const int32_t *k_hubs; int32_t k_n_hubs;
    const int32_t *common_col; const float *common_w; int32_t n_common; const float *alpha; const uint8_t *row_skip;
    /* tile unions of the k_* form (ptk_gcn_aggregate_tiled); NULL / 0: absent */
    const int32_t *tile_uptr, *tile_ucol; const uint16_t *tile_lidx; int32_t max_union;
} ptk_gcn_csr;

size_t ptk_gcn_stack_fwd_workspace_bytes(int64_t B, int64_t Nv, int32_t n_layers, const int64_t *widths,
                                         const int32_t *Ls);
int ptk_gcn_stack_fwd(const ptk_gcn_csr *graph, int64_t B, int64_t Nv, int32_t n_layers, const int64_t *widths,
                      const int32_t *Ls, const uint8_t *relus, const float *X, const float *const *W,
                      const float *const *bias, float *const *acts, uint32_t *const *x_bits, int algo, int fuse,
                      void *workspace, size_t workspace_bytes, ptk_stream_t stream);
/* Backward of the same stack.  graph_t: the TRANSPOSED adjacency.  X, W, acts, x_bits as in the forward; gout
 * (B,Nv,width[n]) the gradient of the last output.  Outputs: gX (B,Nv,width[0]) or NULL; gW[l] (width[l] x width[l+1])
 * or NULL per layer; gb[l] (width[l+1]) where need_gb[l] != 0.  batch_bias != 0: the layers that share the hidden
 * width keep their output gradients in one slab and their bias gradients are two launches in total -- this needs
 * their gb[] pointers to be consecutive rows of one (count x width) matrix, otherwise it falls back to per-layer
 * bias gradients.  algo_dgrad / algo_wgrad: PTK_GEMM_*. */
size_t ptk_gcn_stack_bwd_workspace_bytes(int64_t B, int64_t Nv, int32_t n_layers, const int64_t *widths,
                                         const int32_t *Ls, const uint8_t *need_gb, int batch_bias);
int ptk_gcn_stack_bwd(const ptk_gcn_csr *graph_t, int64_t B, int64_t Nv, int32_t n_layers, const int64_t *widths,
                      const int32_t *Ls, const uint8_t *relus, const float *X, const float *const *W,
                      const float *const *acts, const uint32_t *const *x_bits, const float *gout, float *gX,
                      float *const *gW, float *const *gb, const uint8_t *need_gb, int batch_bias, int algo_dgrad,
                      int algo_wgrad, void *workspace, size_t workspace_bytes, ptk_stream_t stream);

/* ------------------------------------------------------------------------------------------------
 * Max over the vertices: (B,Nv,C) -> out (B,C) and arg (B,C) int32 (may be NULL), lowest vertex id on
 * ties, NaN propagates.  Replaces `features.max(dim=1)[0]` after the GCN encoder of the autoencoder
 * (pterotactyl/reconstruction/autoencoder/model.py:91) and `torch.max(x, dim=1)[0]` of the DDQN
 * Graph_Model (pterotactyl/policies/DDQN/model.py:128).  bwd overwrites grad_in (B,Nv,C):
 * grad_in[b, arg[b,c], c] = grad_out[b,c], zero elsewhere.
 * ---------------------------------------------------------------------------------------------- */
int ptk_vertex_maxpool_fwd(const float *in, int64_t B, int64_t Nv, int64_t C, float *out, int32_t *arg,
                           ptk_stream_t stream);
int ptk_vertex_maxpool_bwd(const float *grad_out, const int32_t *arg, int64_t B, int64_t Nv, int64_t C,
                           float *grad_in, ptk_stream_t stream);

/* ------------------------------------------------------------------------------------------------
 * GCN adjacency built on the device and emitted as CSR -- no dense (Nv,Nv) matrix, no host loops.
 * Replaces calc_adj (pterotactyl/utility/utils.py:134-148: identity + the 6 directed edges of every
 * face), the fusing step of adj_fuse_touch (utils.py:75-130: vertices whose 3-D positions are byte-
 * identical are linked to each other and, both ways, to every touch-chart centre) and normalize_adj
 * (utils.py:47-52: every entry of row i is fl32(1/deg_i)).
 *   faces      (F,3) int32 vertex ids in [0,n) -- for the fused graph: vision faces followed by the
 *              touch-chart faces already offset into the fused numbering
 *   positions  (n_pos,3) f32 positions of vertices 0..n_pos-1 compared for byte equality, or NULL / 0
 *   centres    (n_centres) int32 ids linked to every vertex that has a twin, or NULL / 0
 * ptk_adj_count fills rowptr (n+1) int32 and keeps the edge bitmap + degrees in `workspace`
 * (ptk_adj_workspace_bytes(n); n <= 65536, else 0 / PTK_ERR_SHAPE); the caller reads rowptr[n],
 * allocates col / val / val_t with that many entries and calls ptk_adj_emit with the same workspace.
 * Column ids ascend within a row.  val[k] = 1/deg[row]; val_t[k] = 1/deg[col[k]] are the values of the
 * transposed CSR (the pattern is symmetric, so rowptr and col serve both directions); either may be NULL.
 * ---------------------------------------------------------------------------------------------- */
size_t ptk_adj_workspace_bytes(int64_t n);
int ptk_adj_count(const int32_t *faces, int64_t F, int64_t n, const float *positions, int64_t n_pos,
                  const int32_t *centres, int64_t n_centres, int32_t *rowptr, void *workspace,
                  size_t workspace_bytes, ptk_stream_t stream);
int ptk_adj_emit(int64_t n, const int32_t *rowptr, int32_t *col, float *val, float *val_t,
                 const void *workspace, size_t workspace_bytes, ptk_stream_t stream);

/* ------------------------------------------------------------------------------------------------
 * NeRF positional embedding of vertex positions, fused with the concatenation of the raw positions:
 * positions (M,3) -> out (M,63), row = [sin(s_0 p), cos(s_0 p), ..., sin(s_9 p), cos(s_9 p), p] with
 * s_0 = fl32(pi), s_i = fl32(pi*2*i).  Replaces Positional_Encoder.nerf_embedding + torch.cat
 * (pterotactyl/reconstruction/vision/model.py:381-391, 396-397; ~45 launches per call).  bwd overwrites
 * grad_positions (M,3) from grad_out (M,63).
 * ---------------------------------------------------------------------------------------------- */
int ptk_nerf_embed_fwd(const float *positions, int64_t M, float *out, ptk_stream_t stream);
int ptk_nerf_embed_bwd(const float *positions, const float *grad_out, int64_t M, float *grad_positions,
                       ptk_stream_t stream);

/* ------------------------------------------------------------------------------------------------
 * Vertex-feature front of the deformation network in one launch (csrc/vertex_front.cu):
 *   out (M,width) = Linear3(relu(Linear2(relu(Linear1(nerf_embed(positions)))))) + emb[(int)mask] + add
 * Replaces Positional_Encoder.forward (pterotactyl/reconstruction/vision/model.py:393-399: embedding + cat +
 * Linear(63,h1)+ReLU, Linear(h1,h2)+ReLU, Linear(h2,width)), Mask_Encoder.forward (model.py:410-414: Embedding(4,
 * width) of mask.long()) and the feature additions of Deformation.forward (model.py:234-236, 266-267, 277-279).
 * Weights in nn.Linear layout (out,in) row-major; mask (M) floats (truncated like .long(), clamped to 0..3), emb
 * (4,width) and add (M,width) may be NULL.  h1 <= 112, h2 <= 224.  h1_save (M,h1) / h2_save (M,h2), when given,
 * receive the hidden activations (after ReLU) for the backward.
 * ptk_vertex_front_colsum: sums (4,width), sums[t][n] = sum of g[m][n] over rows whose mask token is t (all rows
 * count as token 0 when mask is NULL) -- the gradient of the embedding table; its column total is the gradient of
 * the last bias.  Fixed-order two-stage reduction (deterministic).
 * ---------------------------------------------------------------------------------------------- */
int ptk_vertex_front_fwd(const float *positions, const float *mask, const float *w1, const float *b1,
                         const float *w2, const float *b2, const float *w3, const float *b3, const float *emb,
                         const float *add, int64_t M, int32_t h1, int32_t h2, int32_t width, float *out,
                         float *h1_save, float *h2_save, ptk_stream_t stream);
size_t ptk_vertex_front_colsum_workspace_bytes(int64_t M, int32_t width);
int ptk_vertex_front_colsum(const float *g, const float *mask, int64_t M, int32_t width, float *sums,
                            void *workspace, size_t workspace_bytes, ptk_stream_t stream);

/* ------------------------------------------------------------------------------------------------
 * utils.chamfer_distance(verts, faces, gt_points, num, repeat) (pterotactyl/utility/utils.py:204-217) on device
 * pointers, one call per pass: repeat x (ptk_sample_fwd -> ptk_chamfer_fwd), cd (B) = the mean over the repeats
 * (sum in repeat order, one multiply by 1/repeat -- torch.stack(cds).mean(0)); backward: repeat x (ptk_chamfer_bwd ->
 * ptk_sample_bwd) accumulated in repeat order.  u_face (repeat,B,S) / uv (repeat,2,B,S): the uniform draws of the
 * repeats in consumption order; u_face may be NULL, face_idx (repeat,B,S) is then the caller's draw (see
 * ptk_sample_fwd).  pts (repeat,B,S,3), face_idx, idx_x (repeat,B,S), idx_y (repeat,B,P2) are what the backward
 * needs.  grad_verts (B,V,3) / grad_gt (B,P2,3) are overwritten; either may be NULL (autoencoder: only grad_gt,
 * autoencoder/train.py:145-150).  workspace: 256-byte aligned, ptk_mesh_chamfer_workspace_bytes.
 * ---------------------------------------------------------------------------------------------- */
size_t ptk_mesh_chamfer_workspace_bytes(int64_t B, int64_t V, int64_t F, int64_t S, int64_t P2);
int ptk_mesh_chamfer_fwd(const float *verts, int64_t B, int64_t V, const int32_t *faces, int64_t F, const float *gt,
                         int64_t P2, const float *u_face, const float *uv, int64_t S, int64_t repeat, float *cd,
                         float *pts, int32_t *face_idx, int32_t *idx_x, int32_t *idx_y, void *workspace,
                         size_t workspace_bytes, ptk_stream_t stream);
int ptk_mesh_chamfer_bwd(const float *gt, const float *pts, const int32_t *face_idx, const int32_t *idx_x,
                         const int32_t *idx_y, const float *uv, const int32_t *faces, const float *grad_cd, int64_t B,
                         int64_t V, int64_t F, int64_t S, int64_t P2, int64_t repeat, float *grad_verts,
                         float *grad_gt, void *workspace, size_t workspace_bytes, ptk_stream_t stream);

/* ------------------------------------------------------------------------------------------------
 * Host-buffer entry points (end-to-end path: H2D + kernels + D2H inside the call).
 * All pointers are HOST pointers (pinned memory makes the copies asynchronous and faster).
 * ---------------------------------------------------------------------------------------------- */
typedef struct ptk_host_ctx ptk_host_ctx;
ptk_host_ctx *ptk_host_ctx_create(int device);
void ptk_host_ctx_destroy(ptk_host_ctx *ctx);
/* Chamfer forward (+ backward when grad_cham != NULL) on host clouds.  cham (B) required;
 * idx_x/idx_y/grad_x/grad_y may be NULL (with grad_cham given the backward still runs on the device;
 * gradients are copied back only where a host pointer is supplied). */
int ptk_host_chamfer(ptk_host_ctx *ctx, const float *x, const float *y, int64_t B, int64_t P1,
                     int64_t P2, float *cham, int32_t *idx_x, int32_t *idx_y, const float *grad_cham,
                     float *grad_x, float *grad_y);
/* utils.chamfer_distance(verts, faces, gt_points, num, repeat) (utils.py:204-217) on host buffers:
 * u_face (repeat,B,S), uv (repeat,2,B,S); cd (B) = mean over repeats; grad_verts (B,V,3) (optional)
 * is d(sum_b grad_cd[b]*cd[b])/d verts. */
int ptk_host_mesh_chamfer(ptk_host_ctx *ctx, const float *verts, int64_t B, int64_t V,
                          const int32_t *faces, int64_t F, const float *gt, int64_t P2,
                          const float *u_face, const float *uv, int64_t S, int64_t repeat, float *cd,
                          const float *grad_cd, float *grad_verts);

#ifdef __cplusplus
}
#endif
#endif /* PTK_H_ */
