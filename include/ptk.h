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

/* Deterministic backward: the gradient of ptk_chamfer_bwd_lengths (same arguments, lengths and reductions), with
 * bits that depend on neither the scheduling nor the batch the pair is computed in.  (The default backward scatters
 * with fp32 atomics: its low bits vary from run to run.)  Per pair b:
 *   - terms: a valid query's own term is s * (q - t[idx]) per component (s = 2 g[b] / max(len, 1) for mean, 2 g[b]
 *     for sum), with the default kernels' fp32 operations; it goes to the query's row and, negated, to its nearest
 *     neighbour's row.  Both directions always take part, so grad_y has the same bits with or without grad_x;
 *   - scale: M_b = the largest finite |term| of both directions, e_b = 62 - ceil(log2 M_b) - ceil(log2(max(lx, ly) + 1));
 *   - rounding: each finite term is quantised to round_half_even(term * 2^e_b) (int64), a row's quantised terms are
 *     summed exactly (no overflow: a row holds at most max(lx, ly) + 1 terms) and the gradient is
 *     ldexpf((float)sum, -e_b): one round-to-nearest-even of the exact quantised sum;
 *   - non-finite terms (NaN / Inf input, overflow of the product) are added to their rows outside the integer sum: a
 *     row with any is NaN if one is NaN or both infinities occur, otherwise that infinity;
 *   - zero rows: padded rows, rows of a pair whose other cloud is empty and every row of a pair with M_b = 0 are +0.
 * grad_x / grad_y (either may be NULL) are fully overwritten.  workspace: 16-byte aligned,
 * ptk_chamfer_bwd_det_workspace_bytes(B, P1, P2) (0 for an empty shape).  PTK_ERR_SHAPE for a null cloud / index /
 * grad_cham pointer or an unknown reduction, PTK_ERR_WORKSPACE for a missing or too small workspace.  Three kernels
 * and a memset, no host synchronisation, capture-safe. */
size_t ptk_chamfer_bwd_det_workspace_bytes(int64_t B, int64_t P1, int64_t P2);
int ptk_chamfer_bwd_det(const float *x, const float *y, const int64_t *len_x, const int64_t *len_y, const int32_t *idx_x,
                        const int32_t *idx_y, const float *grad_cham, int64_t B, int64_t P1, int64_t P2, int reduction,
                        float *grad_x, float *grad_y, void *workspace, size_t workspace_bytes, ptk_stream_t stream);

/* Chamfer normal term: the cham_normals of pytorch3d.loss.chamfer_distance(x, y, x_lengths, y_lengths, x_normals,
 * y_normals, point_reduction=...) of PyTorch3D 0.5.0, on the idx_x / idx_y of ptk_chamfer_fwd_lengths (cham itself is
 * that call's, unchanged).  x_normals (B,P1,3), y_normals (B,P2,3); len_x / len_y as for the ragged calls above.  For
 * pair b write lx = len_x[b], ly = len_y[b] (clamped to [0, P]).  For a valid query x_i (i < lx) with ly > 0 and
 * j = idx_x[b,i], a = x_normals[b,i], n = y_normals[b,j]:
 *     c_i = sum_k (a_k / max(|a|, 1e-6)) * (n_k / max(|n|, 1e-6))     (torch's F.cosine_similarity, eps = 1e-6: each
 *     term_x[b,i] = 1 - |c_i|                                          norm clamped on its own)
 *   - a valid query whose target cloud is empty (ly = 0) reads PyTorch3D's zero-filled gathered normal: c = 0 and the
 *     term is 1 (NaN for a non-finite a, as there);
 *   - padded queries (i >= lx) have term 0; the y direction is the same with idx_y and the roles swapped;
 *   - PTK_REDUCE_MEAN: cham_normals[b] = sum term_x / max(lx, 1) + sum term_y / max(ly, 1) (the divisors of cham);
 *     PTK_REDUCE_SUM: the plain sum.  The sum of a pair is a fixed-order function of the pair alone: its bits depend
 *     neither on the batch nor on the padding it is computed in;
 *   - term_x (B,P1) / term_y (B,P2) (either may be NULL) receive the per-query terms, 0 at padded entries.
 * Padding (normals and idx of padded rows) is never read.  workspace: ptk_chamfer_normals_workspace_bytes(B, P1, P2)
 * of 16-byte aligned slice partials, 0 (workspace may be NULL) up to 16384 points per cloud.  PTK_ERR_SHAPE for a null
 * normals / idx / cham_normals pointer, an unknown reduction, an empty or too large shape or B > 65535;
 * PTK_ERR_WORKSPACE / PTK_ERR_ALIGN for a missing, too small or misaligned workspace.  One kernel (two when the clouds
 * are sliced), PDL-chained, no host synchronisation, capture-safe. */
size_t ptk_chamfer_normals_workspace_bytes(int64_t B, int64_t P1, int64_t P2);
int ptk_chamfer_normals_fwd(const float *x_normals, const float *y_normals, const int64_t *len_x, const int64_t *len_y,
                            const int32_t *idx_x, const int32_t *idx_y, int64_t B, int64_t P1, int64_t P2, int reduction,
                            float *term_x, float *term_y, float *cham_normals, void *workspace, size_t workspace_bytes,
                            ptk_stream_t stream);
/* Gradient of cham_normals under grad_cham_normals (B) w.r.t. the normals only (the points get none: idx is piecewise
 * constant).  It is torch's autograd of the formula above: d|c|/dc = sign(c) with sign(0) = 0, and
 * dc/da = (n / |n|_c - c * a / |a|) / |a|_c, |.|_c the clamped norm, a / |a| = 0 at a = 0.  Each valid query with a
 * non-empty target cloud has an own part, -s sign(c) dc/da onto its normal row, and a near part, -s sign(c) dc/dn onto
 * the gathered row j (s = g[b] / lq for mean, g[b] for sum).  Padded rows, and every row of a pair with lx = 0 or
 * ly = 0 in the direction that has no target, get +0.  grad_xn (B,P1,3) / grad_yn (B,P2,3) (either may be NULL) are
 * fully overwritten; neither requested: return 0 at once.  PTK_ERR_SHAPE as for the forward and for a null
 * grad_cham_normals pointer.  No host synchronisation, capture-safe.
 * ptk_chamfer_normals_bwd: two kernels, the own parts as plain stores, then the near parts with fp32 atomics (their
 * rows' low bits vary from run to run).
 * ptk_chamfer_normals_bwd_det: the scheme of ptk_chamfer_bwd_det per pair: M_b = the largest finite |part| of both
 * directions, e_b = 62 - ceil(log2 M_b) - ceil(log2(max(lx, ly) + 1)) (a row holds one own part and at most l_other
 * near parts), exact int64 sums of round_half_even(part * 2^e_b), grad = ldexpf((float)sum, -e_b), non-finite parts
 * outside the integer sum.  Bits depend neither on scheduling nor on the batch or the order of the queries.  workspace:
 * ptk_chamfer_bwd_det_workspace_bytes(B, P1, P2) (the same layout), 16-byte aligned; PTK_ERR_WORKSPACE when missing or
 * too small.  A memset and three kernels. */
int ptk_chamfer_normals_bwd(const float *x_normals, const float *y_normals, const int64_t *len_x, const int64_t *len_y,
                            const int32_t *idx_x, const int32_t *idx_y, const float *grad_cham_normals, int64_t B,
                            int64_t P1, int64_t P2, int reduction, float *grad_xn, float *grad_yn, ptk_stream_t stream);
int ptk_chamfer_normals_bwd_det(const float *x_normals, const float *y_normals, const int64_t *len_x,
                                const int64_t *len_y, const int32_t *idx_x, const int32_t *idx_y,
                                const float *grad_cham_normals, int64_t B, int64_t P1, int64_t P2, int reduction,
                                float *grad_xn, float *grad_yn, void *workspace, size_t workspace_bytes,
                                ptk_stream_t stream);

/* 1-NN backward: the gradient of dist = ptk_knn1_fwd_lengths(p1, p2, len1, len2) under a per-query upstream gradient
 * grad_dist (B,P1), with the forward's idx (B,P1).  len1 / len2 as above (NULL: full).  For a valid query i < l1[b]
 * of a pair with l2[b] > 0 and j = idx[b,i], the term is t = s * (p1[b,i] - p2[b,j]) per component, s = 2 grad_dist[b,i]
 * (fp32, the operations of PyTorch3D's knn_points_backward for norm 2):
 *   - grad_p1[b,i] = t (a plain store: a p1 row holds exactly one term);
 *   - grad_p2[b,j] -= t, summed over every query that chose j;
 *   - padded queries and queries whose target cloud is empty contribute nothing: their grad_dist is never read, so a
 *     NaN there does not leak.  Padded rows of both gradients, and every row of a pair with l1 = 0 or l2 = 0, are +0.
 * grad_p1 / grad_p2 (either may be NULL) are fully overwritten; neither requested: return 0 at once.  PTK_ERR_SHAPE for
 * a null cloud / idx / grad_dist pointer, an empty or too large shape, B > 65535.  No host synchronisation,
 * capture-safe.  Replaces pytorch3d.ops.knn_points' backward (_C.knn_points_backward) for K = 1.
 * ptk_knn1_bwd_lengths: two kernels, grad_p1 and zeroed grad_p2 rows, then a scatter with fp32 atomics (grad_p2's low
 * bits vary from run to run). */
int ptk_knn1_bwd_lengths(const float *p1, const float *p2, const int64_t *len1, const int64_t *len2, const int32_t *idx,
                         const float *grad_dist, int64_t B, int64_t P1, int64_t P2, float *grad_p1, float *grad_p2,
                         ptk_stream_t stream);
/* Deterministic form: the scheme of ptk_chamfer_bwd_det per pair b.  grad_p1 is the same plain store, with the same
 * bits as ptk_knn1_bwd_lengths.  grad_p2: M_b = the largest finite |term| of the pair's valid queries,
 * e_b = 62 - ceil(log2 M_b) - ceil(log2(l1 + 1)) (a p2 row receives at most l1 terms), exact int64 sums of
 * round_half_even(term * 2^e_b), grad_p2 = ldexpf((float)sum, -e_b); non-finite terms bypass the integer sum as in
 * ptk_chamfer_bwd_det.  Bits depend neither on scheduling nor on the batch the pair runs in.  workspace: 16-byte aligned,
 * ptk_knn1_bwd_det_workspace_bytes(B, P1, P2) = [M_b bits, padded to 256 B][24 B per p2 point] (0 for an empty shape),
 * also required when only grad_p1 is requested; PTK_ERR_WORKSPACE when missing or too small.  A memset and three
 * kernels (one kernel without grad_p2). */
size_t ptk_knn1_bwd_det_workspace_bytes(int64_t B, int64_t P1, int64_t P2);
int ptk_knn1_bwd_det(const float *p1, const float *p2, const int64_t *len1, const int64_t *len2, const int32_t *idx,
                     const float *grad_dist, int64_t B, int64_t P1, int64_t P2, float *grad_p1, float *grad_p2,
                     void *workspace, size_t workspace_bytes, ptk_stream_t stream);

/* K nearest neighbours, 1 <= K <= PTK_KNN_MAX_K: pytorch3d.ops.knn_points(p1, p2, lengths1, lengths2, K).
 * len1 / len2 as for the ragged calls above (device int64, NULL: full, clamped on the device).  For pair b write
 * l1 = len1[b], l2 = len2[b].  For a valid query i < l1, dist[b,i,:] / idx[b,i,:] (B,P1,K) f32 / int32 are the K
 * smallest (d, j) over targets j < l2 in lexicographic order: ascending distance, the lower index first on equal
 * distances.  d is the defining arithmetic of ptk_knn1_fwd (fma(dz,dz, fma(dy,dy, dx*dx)), dx = q.x - t.x).
 * Operationally: K slots of (+inf, 0); j ascending; (d, j) enters when d < slot[K-1].d (strict: an equal distance
 * never displaces a lower index, a NaN or +inf distance never enters) and is inserted after every slot whose distance
 * is <= d.  This is the selection rule of PyTorch3D's knn_cpu.cpp.  Consequences:
 *   - column 0 is ptk_knn1_fwd_lengths' result bit for bit, for every input (NaN, Inf, ties included);
 *   - slots that no finite distance fills stay (+inf, 0);
 *   - zero fill, as PyTorch3D pads: slots k >= l2 are (0, 0), padded queries i >= l1 are (0, 0) in every slot, and
 *     so is every slot of a pair with l2 = 0.  K > P2 is allowed;
 *   - the result is a pure function of the pair: it depends neither on the batch nor on how the target range is split.
 * workspace: 16-byte aligned, ptk_knn_workspace_bytes(B, P1, P2, K) (a function of the shapes only; 0 when the target
 * range is not split, and then workspace may be NULL).  PTK_ERR_SHAPE for a null cloud / dist / idx pointer, an empty
 * or too large shape, B > 65535 or K outside [1, PTK_KNN_MAX_K]; PTK_ERR_WORKSPACE for a missing or too small
 * workspace, PTK_ERR_ALIGN for a misaligned one.  One scan kernel (plus a merge kernel when the target range is
 * split), PDL-chained, no host synchronisation, capture-safe. */
#define PTK_KNN_MAX_K 64
size_t ptk_knn_workspace_bytes(int64_t B, int64_t P1, int64_t P2, int64_t K);
int ptk_knn_fwd_lengths(const float *p1, const float *p2, const int64_t *len1, const int64_t *len2, int64_t B,
                        int64_t P1, int64_t P2, int64_t K, float *dist, int32_t *idx, void *workspace,
                        size_t workspace_bytes, ptk_stream_t stream);
/* K-NN backward: the gradient of dist = ptk_knn_fwd_lengths(...) under the upstream gradient grad_dist (B,P1,K), with
 * the forward's idx (B,P1,K).  Slot k < min(K, l2) of a valid query i < l1, with j = idx[b,i,k], has the term
 * t = s * (p1[b,i] - p2[b,j]) per component, s = 2 grad_dist[b,i,k] (fp32: the operations of ptk_knn1_bwd_lengths and
 * of PyTorch3D's knn_points_backward).  No other slot exists: its grad_dist is never read, so a NaN there does not leak.
 *   - grad_p1[b,i] = the terms of row i summed in slot order, ((t0 + t1) + t2) + ..., in fp32 (no atomics: the same
 *     bits in both forms below);
 *   - grad_p2[b,j] = minus the sum of the terms that chose j;
 *   - padded rows of both gradients, and every row of a pair with l1 = 0 or l2 = 0, are +0.
 * grad_p1 / grad_p2 (either may be NULL) are fully overwritten; neither requested: return 0 at once.  PTK_ERR_SHAPE as
 * for ptk_knn_fwd_lengths and for a null idx / grad_dist pointer.  No host synchronisation, capture-safe.
 * ptk_knn_bwd_lengths: two kernels, grad_p1 with zeroed grad_p2 rows, then a scatter with fp32 atomics (grad_p2's low
 * bits vary from run to run). */
int ptk_knn_bwd_lengths(const float *p1, const float *p2, const int64_t *len1, const int64_t *len2, const int32_t *idx,
                        const float *grad_dist, int64_t B, int64_t P1, int64_t P2, int64_t K, float *grad_p1,
                        float *grad_p2, ptk_stream_t stream);
/* Deterministic form: the scheme of ptk_knn1_bwd_det per pair b.  grad_p1 as above.  grad_p2: M_b = the largest finite
 * |term| of the pair's slots, e_b = 62 - ceil(log2 M_b) - ceil(log2(l1 + 1)) (a query's K indices are distinct, so a p2
 * row receives at most l1 terms), exact int64 sums of round_half_even(term * 2^e_b), grad_p2 = ldexpf((float)sum,
 * -e_b); non-finite terms bypass the integer sum.  Bits depend neither on scheduling nor on the batch or the order of
 * the queries.  workspace: 16-byte aligned, ptk_knn1_bwd_det_workspace_bytes(B, P1, P2) (the same layout), also
 * required when only grad_p1 is requested; PTK_ERR_WORKSPACE when missing or too small.  A memset and three kernels
 * (one kernel without grad_p2). */
int ptk_knn_bwd_det(const float *p1, const float *p2, const int64_t *len1, const int64_t *len2, const int32_t *idx,
                    const float *grad_dist, int64_t B, int64_t P1, int64_t P2, int64_t K, float *grad_p1, float *grad_p2,
                    void *workspace, size_t workspace_bytes, ptk_stream_t stream);

/* Point-cloud normals and local coordinate frames: pytorch3d.ops.estimate_pointcloud_normals and
 * estimate_pointcloud_local_coord_frames of PyTorch3D 0.5.0 (points_normals.py), on idx / dist (B,P,K) of
 * ptk_knn_fwd_lengths(points, points, lengths, lengths, K).  points (B,P,3); lengths as for the ragged calls above.
 * For cloud b write l = lengths[b] and K' = min(K, l).  For a valid query i < l, with q_k = points[b, idx[b,i,k]]:
 *     d_k = q_k - p_i,  m = (1/K') sum_{k<K'} d_k,  C = (1/K') sum_{k<K'} (d_k - m)(d_k - m)^T
 * (the covariance of the neighbours about their mean, computed relative to the query: C is translation invariant).
 * The eigenpairs (lam_m, v_m) of C, lam_0 <= lam_1 <= lam_2, come from a cyclic Jacobi solver with a fixed number of
 * sweeps (so NaN input cannot make it loop); v_0 is normalised, v_2 orthogonalised against it and normalised, and
 * v_1 = v_2 x v_0.  curvatures[b,i] = (lam_0, lam_1, lam_2).
 *   - disambiguate != 0 (PyTorch3D's default): for v in {v_0, v_2}, n_pos = #{k < K' : v . d_k > 0}; v is negated when
 *     n_pos < 0.5 K'.  This gives n (from v_0) and z (from v_2); y = n x z and frames[b,i] has the columns (n, y, z).
 *   - disambiguate == 0: frames[b,i] has the columns (v_0, v_1, v_2) with the solver's signs.
 *   - normals[b,i] = frames[b,i][:, 0], bit for bit; frames[b,i,r,c] is component r of column c.
 *   - repeated eigenvalues (C = 0 at K' = 1, exactly planar or collinear neighbourhoods): any orthonormal basis of the
 *     eigenspace; the result is still finite, unit-length, orthonormal and a deterministic function of the input.
 *   - padded queries (i >= l): every output is 0.
 *   - a query with a slot k < K' whose distance is not finite (a NaN / Inf point, or a slot left at (+inf, 0) by the
 *     K-NN) gets NaN in every output.  A NaN point never enters another query's neighbourhood, so it changes nothing
 *     else.  l <= K is not an error (K' handles it) and needs no host synchronisation.
 * ptk_point_frames_fwd writes normals (may be NULL) and / or curvatures (B,P,3) with frames (B,P,3,3) (both NULL or
 * both given); at least one output.  One kernel, one thread per query, PDL-chained, capture-safe.
 * PTK_ERR_SHAPE for a null points / idx / dist / output pointer, an empty or too large shape, B > 65535 or K outside
 * [1, PTK_KNN_MAX_K]. */
int ptk_point_frames_fwd(const float *points, const int64_t *lengths, const int32_t *idx, const float *dist, int64_t B,
                         int64_t P, int64_t K, int disambiguate, float *normals, float *curvatures, float *frames,
                         ptk_stream_t stream);
/* Gradient of the outputs above w.r.t. points under grad_normals (B,P,3), grad_curvatures (B,P,3) and grad_frames
 * (B,P,3,3), any of which may be NULL (zero).  The eigensystem is recomputed with the forward's arithmetic; nothing but
 * the inputs is saved.  Per valid query, gV folds the upstream gradients into the eigenvectors: with disambiguate,
 * g_n += z x g_y and g_z += g_y x n (y = n x z), then g_v0 = s_0 g_n and g_v2 = s_2 g_z (s = the signs applied);
 * without it g_v0 / g_v1 / g_v2 are the frame columns' gradients.  Normals add to g_n (resp. g_v0).  Then, as
 * torch.linalg.eigh's backward,
 *     G = V (diag(g_lam) + F o (V^T gV)) V^T,  F_mn = 1 / (lam_n - lam_m) for m != n, 0 on the diagonal,
 * where F_mn is taken as 0 when lam_n == lam_m in fp32 (a repeated eigenspace has no defined gradient), and slot k adds
 *     (1/K') (G + G^T) (q_k - mean of the q)
 * to the gradient of point idx[b,i,k].  Terms that are zero analytically are left out: those through the mean (the
 * centred neighbours sum to zero), through the query's own p_i (C is translation invariant) and through the sign rule
 * (a step function).  Padded queries and queries with NaN outputs pass no gradient.  grad_points (B,P,3) is fully
 * overwritten; padded rows are +0.  PTK_ERR_SHAPE as for the forward and for a null grad_points pointer.  No host
 * synchronisation, capture-safe.
 * ptk_point_frames_bwd: a memset and one kernel, the terms added with fp32 atomics (low bits vary from run to run).
 * ptk_point_frames_bwd_det: the scheme of ptk_knn_bwd_det per cloud b: M_b = the largest finite |term|,
 * e_b = 62 - ceil(log2 M_b) - ceil(log2(l + 1)) (a query's K' indices are distinct, so a point receives at most l
 * terms), exact int64 sums of round_half_even(term * 2^e_b), grad = ldexpf((float)sum, -e_b); non-finite terms bypass
 * the integer sum.  Bits depend neither on scheduling nor on the batch or the order of the points.  workspace:
 * 16-byte aligned, ptk_knn1_bwd_det_workspace_bytes(B, P, P) (the same layout); PTK_ERR_WORKSPACE when missing or too
 * small, PTK_ERR_ALIGN when misaligned.  A memset and three kernels. */
int ptk_point_frames_bwd(const float *points, const int64_t *lengths, const int32_t *idx, const float *dist, int64_t B,
                         int64_t P, int64_t K, int disambiguate, const float *grad_normals, const float *grad_curvatures,
                         const float *grad_frames, float *grad_points, ptk_stream_t stream);
int ptk_point_frames_bwd_det(const float *points, const int64_t *lengths, const int32_t *idx, const float *dist,
                             int64_t B, int64_t P, int64_t K, int disambiguate, const float *grad_normals,
                             const float *grad_curvatures, const float *grad_frames, float *grad_points,
                             void *workspace, size_t workspace_bytes, ptk_stream_t stream);

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
/* Deterministic ptk_sample_bwd, the scheme of ptk_chamfer_bwd_det per mesh b: the terms are c = w_k * grad_pts[b,s,d]
 * (the default kernel's fp32 operations), M_b = the largest finite |c|, e_b = 62 - ceil(log2 M_b) - ceil(log2(3 S + 1))
 * (a vertex receives at most 3 S terms: a degenerate face may list it twice), exact int64 sums of
 * round_half_even(c * 2^e_b), grad = ldexpf((float)sum, -e_b); non-finite terms as in ptk_chamfer_bwd_det; vertices
 * no sample touches (and every vertex when M_b = 0) are +0.  grad_verts is fully overwritten.  workspace: 16-byte
 * aligned, ptk_sample_bwd_det_workspace_bytes(B, V) (0 for an empty shape). */
size_t ptk_sample_bwd_det_workspace_bytes(int64_t B, int64_t V);
int ptk_sample_bwd_det(const float *grad_pts, const int32_t *face_idx, const float *uv, const int32_t *faces, int64_t B,
                       int64_t V, int64_t F, int64_t S, float *grad_verts, void *workspace, size_t workspace_bytes,
                       ptk_stream_t stream);

/* Normals of the sampled points: the return_normals branch of PyTorch3D 0.5.0's sample_points_from_meshes
 * ((v1 - v0).cross(v2 - v1), divided by its norm clamped to at least sys.float_info.epsilon, gathered by the sampled
 * face index), on the face_idx (B,S) of ptk_sample_fwd.  For sample s of mesh b on face f = face_idx[b,s], clamped to
 * [0, F-1] as sample_points_kernel clamps a given index, with corners v0, v1, v2 (fp32, every product, difference and
 * sum rounded on its own, no FMA contraction, as in the sampler's face areas):
 *     e1 = v1 - v0,  e2 = v2 - v1             (not the v2 - v0 of ptk_face_areas_normals, which keeps its 1e-6 clamp)
 *     c0 = e1y e2z - e1z e2y,  c1 = e1z e2x - e1x e2z,  c2 = e1x e2y - e1y e2x
 *     r  = sqrt((c0 c0 + c1 c1) + c2 c2)
 *     q  = r < eps ? eps : r                  (eps = 2^-52, the fp32 value of 2.220446049250313e-16; NaN stays NaN)
 *     normals[b,s] = c / q                    (IEEE division)
 * A face with a NaN or Inf vertex gives NaN / Inf normals (no check, no host synchronisation); a degenerate face
 * (r < eps) gives c / eps, (0, 0, 0) when c = 0.  normals (B,S,3) is fully overwritten.  PTK_ERR_SHAPE for a null
 * pointer, an empty or too large shape or B > 65535.  One kernel, PDL-chained after ptk_sample_fwd, capture-safe. */
int ptk_sample_normals_fwd(const float *verts, int64_t B, int64_t V, const int32_t *faces, int64_t F,
                           const int32_t *face_idx, int64_t S, float *normals, ptk_stream_t stream);
/* Gradient of pts = ptk_sample_fwd(...) and normals = ptk_sample_normals_fwd(...) w.r.t. verts, under grad_pts (B,S,3)
 * (may be NULL: a loss on the normals only) and grad_normals (B,S,3).  It is torch's autograd of the formula above.
 * Per sample, with n = c / q and g = grad_normals[b,s]:
 *     g_c = (g - (n . g) n) / q    when r >= eps  (= g / r - (c . g) c / r^3; at r = eps the clamp passes the gradient
 *                                                  through, as clamp_min's backward does)
 *     g_c = g / eps                when r < eps
 *     g_e1 = e2 x g_c,  g_e2 = g_c x e1;  normal terms g_v0 = -g_e1, g_v1 = g_e1 - g_e2, g_v2 = g_e2
 * and the sampler's point terms w_k * grad_pts[b,s] (w: the barycentric weights of ptk_sample_fwd).  One shared
 * device function states the per-sample fp32 operations, so both forms below add the same terms.
 * grad_verts (B,V,3) is fully overwritten; vertices no sample touches are +0.  PTK_ERR_SHAPE for a null pointer (other
 * than grad_pts), an empty or too large shape or B > 65535.  No host synchronisation, capture-safe.
 * ptk_sample_normals_bwd: a memset and one kernel: per (sample, corner, component) the point and normal terms are
 * added, then one fp32 atomic, into shared memory for meshes of up to 4096 vertices (then one RED per touched
 * component), straight into grad_verts otherwise (the low bits vary from run to run).
 * ptk_sample_normals_bwd_det: the scheme of ptk_sample_bwd_det per mesh b, with two separately quantised terms per
 * (sample, corner, component): M_b = the largest finite |term| of both kinds, e_b = 62 - ceil(log2 M_b) -
 * ceil(log2(6 S + 1)) (a vertex receives at most 3 S point and 3 S normal terms), exact int64 sums of
 * round_half_even(term * 2^e_b), grad = ldexpf((float)sum, -e_b); non-finite terms outside the integer sum.  Bits
 * depend neither on scheduling nor on the batch or the order of the samples.  Precision is relative to M_b: a
 * degenerate face's terms are of size |g| / eps and swamp the rest of its mesh, as they do in PyTorch3D's own
 * gradient.  workspace: 16-byte aligned, ptk_sample_normals_bwd_det_workspace_bytes(B, V) = [M_b bits, padded to
 * 256 B][24 B per vertex] (0 for an empty shape); PTK_ERR_WORKSPACE when missing or too small, PTK_ERR_ALIGN when
 * misaligned.  A memset and three kernels. */
int ptk_sample_normals_bwd(const float *verts, const int32_t *faces, const int32_t *face_idx, const float *uv,
                           const float *grad_pts, const float *grad_normals, int64_t B, int64_t V, int64_t F, int64_t S,
                           float *grad_verts, ptk_stream_t stream);
size_t ptk_sample_normals_bwd_det_workspace_bytes(int64_t B, int64_t V);
int ptk_sample_normals_bwd_det(const float *verts, const int32_t *faces, const int32_t *face_idx, const float *uv,
                               const float *grad_pts, const float *grad_normals, int64_t B, int64_t V, int64_t F,
                               int64_t S, float *grad_verts, void *workspace, size_t workspace_bytes, ptk_stream_t stream);

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
 * Finite range of the tensor-core paths: operands must satisfy |x| < 2^128 - 2^116 (FLT_MAX is 2^128 - 2^104).
 * From there on, and for +-Inf and NaN, the TF32 split rounds x to +-Inf and its low part becomes NaN, so every
 * output that x reaches is NaN -- where an fp32 loop would give +-Inf (or a finite value).  The FFMA paths follow
 * IEEE fp32.
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
/* The same backward on the deterministic pieces: repeat x (ptk_chamfer_bwd_det -> ptk_sample_bwd_det), accumulated in
 * repeat order as above, so the result is bit-identical to that composition.  workspace: 256-byte aligned,
 * ptk_mesh_chamfer_bwd_det_workspace_bytes (0 for an empty shape). */
size_t ptk_mesh_chamfer_bwd_det_workspace_bytes(int64_t B, int64_t V, int64_t F, int64_t S, int64_t P2);
int ptk_mesh_chamfer_bwd_det(const float *gt, const float *pts, const int32_t *face_idx, const int32_t *idx_x,
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
