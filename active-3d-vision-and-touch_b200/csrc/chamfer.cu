// Chamfer distance / brute-force 1-NN for sm_100a.
//
// Replaces PyTorch3D 0.5.0 KNearestNeighborKernelV3<D=3,K=1> + KNearestNeighborBackwardKernel as
// reached from pterotactyl/utility/utils.py:207,212 (pytorch3d.loss.chamfer_distance).
//
// Design (DESIGN.md "K1"):
//   * FP32-pipe bound.  One distance evaluation = 3 FADD + 1 FMUL + 2 FFMA = 6 FMA-pipe issue slots;
//     everything else is overhead to be amortised:
//       - targets are staged once per CTA in shared memory as SoA (x[], y[], z[]) and read back
//         with 128-bit broadcast loads: 3 LDS.128 per 4 targets, shared by the R queries a thread
//         keeps in registers  => 0.75/R LDS per evaluation;
//       - the running minimum uses the 3-input FMNMX3 of sm_100 (0.5 ALU-pipe op / evaluation);
//       - the arg-min is LAZY: the inner loop only tracks, per query, the minimum over a chunk of
//         16 targets and the id of the first chunk that achieved the running minimum (3 ops per 16
//         evaluations).  The exact index is recovered afterwards by re-evaluating that one chunk
//         with the same instruction sequence (bit-identical distances) and taking the first hit:
//         strict '<' across ascending chunks + first hit inside the chunk == PyTorch3D's
//         "lowest index wins ties".
//   * both directions (x->y and y->x) run in the same launch (blockIdx.z = 2*b + dir).
//   * when the batch is too small to fill 148 SMs the target range is split across CTAs
//     (blockIdx.y) and partial results are merged with a 64-bit atomicMin on the packed key
//     (dist_bits << 32 | idx): dist >= +0 so its bit pattern orders like an unsigned integer and
//     the low word makes the lowest index win ties -- deterministic.
//   * a second small kernel unpacks the keys and does the fused mean reduction in a fixed order
//     (deterministic, no float atomics).
//   * default algorithm (PTK_CHAMFER_FILTER): the scan above is run on the 3-FFMA expansion
//     |t|^2 - 2 q.t with packed FFMA2 instructions as a FILTER (chamfer_kernel2.cuh).  Its target tiles
//     are TMA-staged (cp.async.bulk + mbarrier, double buffered) from padded SoA arrays a small
//     pre-pass writes (chamfer_prep_kernel).  The chunk the filter records is re-evaluated with the
//     defining arithmetic, and the few queries whose runner-up chunk is within the proven error bound
//     are re-scanned exactly (chamfer_nn_exact2_kernel, list mode).  Results are bit-identical to
//     PTK_CHAMFER_EXACT (the 6-op scan on packed FP32x2, kept selectable for checks).
//   * PTK_CHAMFER_PRUNED (chamfer_pruned.cuh): the same results from a cell-sorted copy of both clouds and a box
//     hierarchy -- a few hundred evaluations per query instead of P; PTK_CHAMFER_AUTO picks it for large clouds.
//   * ragged batches (ptk_*_lengths): one code path -- every kernel bounds its queries and targets by the pair's
//     device-side lengths (pair_len(), NULL = full) and keeps the padded strides; the homogeneous calls pass NULL.
#include <atomic>

#include "chamfer_kernel2.cuh"
#include "chamfer_pruned.cuh"

namespace ptk {

// library configuration of the kernel template (tuned with tools/chamfer_tune.cu)
constexpr int CH_THREADS = 128;
constexpr int CH_CHUNK = 16;   // exact scan; filter scan on clouds the recheck cannot read with vector loads
constexpr int CH_CHUNK_F = 64; // filter scan: one bookkeeping step per 64 targets (DESIGN.md K1)
constexpr int CH_WIDE_MIN_SPLIT = 2048;  // fewer targets per split: 16-target chunks (see launch_nn)
constexpr int CH_MINB = 3;   // exact scan
constexpr int CH_MINB_F = 4; // filter scan
constexpr int CH_TT_F = 1024; // targets per TMA tile (double buffered: 2 x 4 x 4 KB)

// process-wide choice of the scan (all give identical results); atomic: other host threads may launch while it is set
static std::atomic<int> g_chamfer_algo{PTK_CHAMFER_AUTO};

// workspace: [PairAux B][soa_x B*4*P1p][soa_y B*4*P2p][stage_x B*4*P1p][stage_y B*4*P2p][box_x B*nbx(P1)][box_y B*nbx(P2)]
//            [keys_x B*P1][keys_y B*P2]
//            [rescue_x B*P1][rescue_y B*P2][flag_x B*P1][flag_y B*P2][count 2B][bad 2B][wide 2B][ghist 2B*bins]
//            (the last two only when the wide sort applies: few large clouds, pr_wide_applies)
//            (P?p = cloud size padded to SOA_PAD points; stage, boxes and `bad` belong to the pruned scan, which also
//            keeps its cell-sorted clouds in soa_x / soa_y)
struct ChamferWs {
    PairAux *aux;
    float *soa_x, *soa_y;
    float4 *stage_x, *stage_y;
    PrBox *box_x, *box_y;
    int *bad;
    PrWide *wide;
    unsigned int *ghist;
    u64 *keys_x, *keys_y;
    int *rescue_x, *rescue_y;
    unsigned int *flag_x, *flag_y, *count;
};

// The wide (multi-launch) sort of the pruned scan: at most 128 clouds, the larger of at least 16k points.  A pure
// function of the sizes: the workspace layout depends on it.
static bool pr_wide_applies(int64_t B, int64_t P1, int64_t P2) { return 2 * B <= 128 && (P1 > P2 ? P1 : P2) >= 16384; }
static bool pr_fine_grid(int64_t P1, int64_t P2) { return (P1 > P2 ? P1 : P2) > 32768; }  // 32^3 cells instead of 16^3
static size_t pr_wide_bytes(int64_t B, int64_t P1, int64_t P2) {
    if (!pr_wide_applies(B, P1, P2)) return 0;
    return (size_t)(2 * B) * (sizeof(PrWide) + 4 * (size_t)(pr_fine_grid(P1, P2) ? 32768 : 4096));
}

static size_t chamfer_ws_bytes(int64_t B, int64_t P1, int64_t P2) {
    return sizeof(PairAux) * (size_t)B + 32 * (size_t)B * (size_t)(soa_padded((int)P1) + soa_padded((int)P2)) +
           sizeof(PrBox) * (size_t)B * (size_t)(pr_boxes((int)P1) + pr_boxes((int)P2)) +
           (size_t)B * (size_t)(P1 + P2) * (8 + 4 + 4) + 16 * (size_t)B + pr_wide_bytes(B, P1, P2);
}

static ChamferWs carve(void *workspace, int64_t B, int64_t P1, int64_t P2) {
    ChamferWs w;
    char *p = reinterpret_cast<char *>(workspace);
    w.aux = reinterpret_cast<PairAux *>(p);
    p += sizeof(PairAux) * (size_t)B;
    w.soa_x = reinterpret_cast<float *>(p);
    p += 16 * (size_t)B * soa_padded((int)P1);
    w.soa_y = reinterpret_cast<float *>(p);
    p += 16 * (size_t)B * soa_padded((int)P2);
    w.stage_x = reinterpret_cast<float4 *>(p);
    p += 16 * (size_t)B * soa_padded((int)P1);
    w.stage_y = reinterpret_cast<float4 *>(p);
    p += 16 * (size_t)B * soa_padded((int)P2);
    w.box_x = reinterpret_cast<PrBox *>(p);
    p += sizeof(PrBox) * (size_t)B * pr_boxes((int)P1);
    w.box_y = reinterpret_cast<PrBox *>(p);
    p += sizeof(PrBox) * (size_t)B * pr_boxes((int)P2);
    w.keys_x = reinterpret_cast<u64 *>(p);
    p += 8 * (size_t)B * P1;
    w.keys_y = reinterpret_cast<u64 *>(p);
    p += 8 * (size_t)B * P2;
    w.rescue_x = reinterpret_cast<int *>(p);
    p += 4 * (size_t)B * P1;
    w.rescue_y = reinterpret_cast<int *>(p);
    p += 4 * (size_t)B * P2;
    w.flag_x = reinterpret_cast<unsigned int *>(p);
    p += 4 * (size_t)B * P1;
    w.flag_y = reinterpret_cast<unsigned int *>(p);
    p += 4 * (size_t)B * P2;
    w.count = reinterpret_cast<unsigned int *>(p);
    p += 8 * (size_t)B;
    w.bad = reinterpret_cast<int *>(p);
    p += 8 * (size_t)B;
    w.wide = reinterpret_cast<PrWide *>(p);
    p += sizeof(PrWide) * (size_t)(2 * B);
    w.ghist = reinterpret_cast<unsigned int *>(p);
    return w;
}

// Unpack keys -> (dist, idx) and reduce the per-cloud sums in a fixed order.
// grid = (B, nsplit), block = 512.  cham may be NULL (plain knn).  nsplit = fin_splits(P1, P2) is a function of the cloud
// sizes only (1 up to 16k points): CTA (b, s) handles slice s of both clouds of pair b; with nsplit > 1 it writes its two
// partial sums to `partial` and chamfer_finalize_sum_kernel adds them in slice order -- deterministic, and a pair's value
// does not depend on the batch it is computed in.  In a ragged batch each pair is sliced by fin_splits of its OWN lengths
// (CTAs past that count only zero-fill padding), so its value is also that of a homogeneous call on the sliced pair.
// Padded queries (i >= len) and queries whose target cloud is empty get dist = 0, idx = 0 (PyTorch3D's zero fill).
constexpr int FIN_SLICE = 16384;
__host__ __device__ inline int fin_splits(int64_t P1, int64_t P2) {
    const int64_t n = ceil_div(P1 > P2 ? P1 : P2, (int64_t)FIN_SLICE);
    return (int)(n < 1 ? 1 : (n > 64 ? 64 : n));
}

// cham[b] from the two sums: mean = sum_x / max(lx, 1) + sum_y / max(ly, 1), sum = sum_x + sum_y
__device__ __forceinline__ float chamfer_reduce(float sx, float sy, int L1, int L2, int mean) {
    return mean ? sx / (float)max(L1, 1) + sy / (float)max(L2, 1) : sx + sy;
}

__global__ void __launch_bounds__(512)
chamfer_finalize_kernel(const unsigned long long *__restrict__ keys_x,
                        const unsigned long long *__restrict__ keys_y, int P1, int P2,
                        const int64_t *__restrict__ len_x, const int64_t *__restrict__ len_y, int mean,
                        float *__restrict__ dist_x, int32_t *__restrict__ idx_x,
                        float *__restrict__ dist_y, int32_t *__restrict__ idx_y,
                        float *__restrict__ cham, float *__restrict__ partial) {
    pdl_wait();  // launched with programmatic stream serialization (ptk_common.cuh)
    const int b = blockIdx.x, sp = blockIdx.y, nsp = gridDim.y;
    const int tid = threadIdx.x;
    const int L1 = pair_len(len_x, b, P1), L2 = pair_len(len_y, b, P2);
    const int nv = fin_splits(L1, L2);  // == nsp without lengths
    __shared__ float red[16];
    float sum[2] = {0.f, 0.f};
    for (int dir = 0; dir < 2; ++dir) {
        const unsigned long long *keys = dir == 0 ? keys_x : keys_y;
        if (keys == nullptr) continue;
        const int P = dir == 0 ? P1 : P2;
        const int L = (dir == 0 ? L2 : L1) == 0 ? 0 : (dir == 0 ? L1 : L2);  // queries with a key; no target: none
        float *dist = dir == 0 ? dist_x : dist_y;
        int32_t *idx = dir == 0 ? idx_x : idx_y;
        float acc = 0.f;
        if (sp < nv) {
            const int len = (int)(((long long)L + nv - 1) / nv), i0 = sp * len, i1 = min(L, i0 + len);
#pragma unroll 8
            for (int i = i0 + tid; i < i1; i += 512) {
                unsigned long long k = keys[(size_t)b * P + i];
                float d = __uint_as_float((unsigned int)(k >> 32));
                if (dist) dist[(size_t)b * P + i] = d;
                if (idx) idx[(size_t)b * P + i] = (int32_t)(unsigned int)(k & 0xffffffffull);
                acc += d;
            }
        }
        const int plen = (P - L + nsp - 1) / nsp, p0 = L + sp * plen, p1 = min(P, p0 + plen);
        for (int i = p0 + tid; i < p1; i += 512) {
            if (dist) dist[(size_t)b * P + i] = 0.f;
            if (idx) idx[(size_t)b * P + i] = 0;
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
    if (tid == 0 && cham) {
        if (nsp == 1) {
            cham[b] = chamfer_reduce(sum[0], sum[1], L1, L2, mean);
        } else if (sp < nv) {
            partial[((size_t)b * nsp + sp) * 2 + 0] = sum[0];
            partial[((size_t)b * nsp + sp) * 2 + 1] = sum[1];
        }
    }
}

// grid = ceil(B / 128), block = 128: cham[b] from the sums of the pair's slice partials, in slice order (a single
// partial p gives 0 + p = p: the value of an unsliced pair)
__global__ void __launch_bounds__(128)
chamfer_finalize_sum_kernel(const float *__restrict__ partial, int B, int nsp, int P1, int P2,
                            const int64_t *__restrict__ len_x, const int64_t *__restrict__ len_y, int mean,
                            float *__restrict__ cham) {
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
    cham[b] = chamfer_reduce(sx, sy, L1, L2, mean);
}

// Backward, phase A (plain stores): the "own point" terms, s_x = 2 g[b] / max(lx, 1) (mean) or 2 g[b] (sum).
//   grad_x[b,i] = s_x * (x_i - y[idx_x[i]]);  grad_y[b,j] = s_y * (y_j - x[idx_y[j]])
// Padded points (i >= len) and points whose target cloud is empty get 0: every row is written.
__global__ void chamfer_bwd_direct_kernel(const float *__restrict__ x, const float *__restrict__ y,
                                          const int32_t *__restrict__ idx_x,
                                          const int32_t *__restrict__ idx_y,
                                          const float *__restrict__ grad_cham, int P1, int P2,
                                          const int64_t *__restrict__ len_x, const int64_t *__restrict__ len_y, int mean,
                                          float *__restrict__ grad_x, float *__restrict__ grad_y) {
    pdl_wait();  // launched with programmatic stream serialization (ptk_common.cuh)
    const int b = blockIdx.y;
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    const float g = grad_cham[b];
    const float *xb = x + (size_t)b * P1 * 3, *yb = y + (size_t)b * P2 * 3;
    const int L1 = pair_len(len_x, b, P1), L2 = pair_len(len_y, b, P2);
    if (grad_x && i < P1) {
        float *o = grad_x + ((size_t)b * P1 + i) * 3;
        if (i < L1 && L2 > 0) {
            const int j = idx_x[(size_t)b * P1 + i];
            const float s = mean ? 2.0f * (g / (float)L1) : 2.0f * g;
            o[0] = s * (xb[i * 3 + 0] - yb[j * 3 + 0]);
            o[1] = s * (xb[i * 3 + 1] - yb[j * 3 + 1]);
            o[2] = s * (xb[i * 3 + 2] - yb[j * 3 + 2]);
        } else {
            o[0] = o[1] = o[2] = 0.f;
        }
    }
    if (grad_y && i < P2) {
        float *o = grad_y + ((size_t)b * P2 + i) * 3;
        if (i < L2 && L1 > 0) {
            const int j = idx_y[(size_t)b * P2 + i];
            const float s = mean ? 2.0f * (g / (float)L2) : 2.0f * g;
            o[0] = s * (yb[i * 3 + 0] - xb[j * 3 + 0]);
            o[1] = s * (yb[i * 3 + 1] - xb[j * 3 + 1]);
            o[2] = s * (yb[i * 3 + 2] - xb[j * 3 + 2]);
        } else {
            o[0] = o[1] = o[2] = 0.f;
        }
    }
}

// Backward, phase B (scatter): the "I am somebody's nearest neighbour" terms, RED.ADD.F32, from valid queries with a
// non-empty target cloud only.
//   grad_y[b, idx_x[i]] -= s_x (x_i - y[idx_x[i]]);  grad_x[b, idx_y[j]] -= s_y (y_j - x[idx_y[j]])
__global__ void chamfer_bwd_scatter_kernel(const float *__restrict__ x, const float *__restrict__ y,
                                           const int32_t *__restrict__ idx_x,
                                           const int32_t *__restrict__ idx_y,
                                           const float *__restrict__ grad_cham, int P1, int P2,
                                           const int64_t *__restrict__ len_x, const int64_t *__restrict__ len_y, int mean,
                                           float *__restrict__ grad_x, float *__restrict__ grad_y) {
    pdl_wait();  // launched with programmatic stream serialization (ptk_common.cuh)
    const int b = blockIdx.y;
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    const float g = grad_cham[b];
    const float *xb = x + (size_t)b * P1 * 3, *yb = y + (size_t)b * P2 * 3;
    const int L1 = pair_len(len_x, b, P1), L2 = pair_len(len_y, b, P2);
    if (grad_y && i < L1 && L2 > 0) {
        const int j = idx_x[(size_t)b * P1 + i];
        const float s = mean ? 2.0f * (g / (float)L1) : 2.0f * g;
        float *o = grad_y + ((size_t)b * P2 + j) * 3;
        atomicAdd(o + 0, -(s * (xb[i * 3 + 0] - yb[j * 3 + 0])));
        atomicAdd(o + 1, -(s * (xb[i * 3 + 1] - yb[j * 3 + 1])));
        atomicAdd(o + 2, -(s * (xb[i * 3 + 2] - yb[j * 3 + 2])));
    }
    if (grad_x && i < L2 && L1 > 0) {
        const int j = idx_y[(size_t)b * P2 + i];
        const float s = mean ? 2.0f * (g / (float)L2) : 2.0f * g;
        float *o = grad_x + ((size_t)b * P1 + j) * 3;
        atomicAdd(o + 0, -(s * (yb[i * 3 + 0] - xb[j * 3 + 0])));
        atomicAdd(o + 1, -(s * (yb[i * 3 + 1] - xb[j * 3 + 1])));
        atomicAdd(o + 2, -(s * (yb[i * 3 + 2] - xb[j * 3 + 2])));
    }
}

// ---------------------------------------------------------------------------------------- host side
struct NNPlan {
    int R;          // queries per thread
    int n_split;    // CTAs along the target range
    int split_len;  // targets per split (multiple of the scan's chunk, so every split starts on a chunk boundary)
};

static NNPlan plan_nn(int64_t B, int64_t Pq_max, int64_t Pt_max, int ndir, int minb, int64_t chunk) {
    // With >= 4 waves of CTAs (minb resident per SM) from the query blocks alone, the target range is not split.
    // Otherwise prefer R = 8 queries per thread (fewest shared-memory loads per evaluation) and get the CTA count
    // from splitting the target range; fall back to fewer queries per thread for tiny clouds.
    const int64_t want = 4LL * sm_count() * minb;
    NNPlan p;
    auto ctas = [&](int R) { return B * ndir * ceil_div(Pq_max, (int64_t)CH_THREADS * R); };
    const int64_t max_split = ceil_div(Pt_max, (int64_t)CH_CHUNK * 16);  // >= 256 targets per split
    p.R = 8;
    if (ctas(8) * max_split < want) p.R = 4;
    if (p.R == 4 && ctas(4) * max_split < want) p.R = 2;
    const int64_t base = ctas(p.R);
    // Splits of the target range: more splits balance the SMs better (the tail of a launch is about one CTA's
    // duration ~ Pt / ns), fewer splits save the fixed cost per CTA (query loads, first tile latency, key merge:
    // ~512 targets' worth, fitted on tools/chamfer_split_sweep.py).  Minimising
    //     (base * ns / slots) * (Pt / ns + 512) + (Pt / ns + 512)      over ns
    // gives ns = sqrt(Pt * slots / (512 * base)); within ~3 % of the measured optimum for P = 4k..100k, B = 1..64.
    const double slots = (double)sm_count() * minb;
    int64_t ns = base >= want ? 1 : (int64_t)(sqrt((double)Pt_max * slots / (512.0 * (double)base)) + 0.5);
    auto split_len = [&](int64_t n) { return ceil_div(ceil_div(Pt_max, n), chunk) * chunk; };
    if (getenv("PTK_CH_NSPLIT")) ns = atoi(getenv("PTK_CH_NSPLIT"));  // tuning tools only (read per call)
    if (ns < 1) ns = 1;
    if (ns > max_split) ns = max_split;
    const int64_t len = split_len(ns);
    p.n_split = (int)ceil_div(Pt_max, len);
    p.split_len = (int)len;
    return p;
}

static unsigned long long g_pr_optin = 0ull;  // cudaFuncAttributeMaxDynamicSharedMemorySize is per device

// PTK_CHAMFER_PRUNED: sort both clouds into cells (one CTA per cloud), walk the box hierarchy (one warp per 32 sorted
// queries), re-scan the queued queries (exact ties across leaves, non-finite clouds) with the exact kernel.
static int launch_nn_pruned(const float *x, const float *y, const int64_t *lx, const int64_t *ly, int64_t B, int64_t P1,
                            int64_t P2, const ChamferWs &w, int dir_only, cudaStream_t st) {
    const int ndir = dir_only >= 0 ? 1 : 2;
    const int64_t Pq = dir_only == 0 ? P1 : (dir_only == 1 ? P2 : (P1 > P2 ? P1 : P2));
    const int64_t Pt = dir_only == 0 ? P2 : (dir_only == 1 ? P1 : (P1 > P2 ? P1 : P2));
    const int iP1 = (int)P1, iP2 = (int)P2;
    PTK_REQUIRE(2 * B <= 0x7fffffffLL && B * ndir <= 65535, PTK_ERR_SHAPE,
                "chamfer: batch %lld too large for one launch (max 32767 clouds)", (long long)B);
    // 16^3 cells up to 32k points (a 16-point leaf then spans about one or two cells), 32^3 above
    const bool fine = pr_fine_grid(P1, P2);
    if (pr_wide_applies(B, P1, P2)) {
        // few large clouds: every phase of the sort is its own launch over slices of all clouds
        const int NC = fine ? 32768 : 4096;
        const int64_t Pm = P1 > P2 ? P1 : P2;
        const dim3 sgrid((unsigned)ceil_div(Pm, (int64_t)PRW_SLICE), (unsigned)(2 * B));
        launch_pdl(pr_wide_init_kernel, dim3((unsigned)(NC / 1024), (unsigned)(2 * B)), dim3(1024), 0, st, w.wide, w.ghist, NC,
                   w.count);
        PTK_CHECK_LAUNCH();
        launch_pdl(pr_wide_bbox_kernel, sgrid, dim3(PRW_THREADS), 0, st, x, y, iP1, iP2, lx, ly, w.wide);
        PTK_CHECK_LAUNCH();
        if (fine) {
            launch_pdl(pr_wide_hist_scatter_kernel<5, false>, sgrid, dim3(PRW_THREADS), 0, st, x, y, iP1, iP2, lx, ly,
                       (const PrWide *)w.wide, w.ghist, w.soa_x, w.soa_y, w.stage_x, w.stage_y, w.bad);
            PTK_CHECK_LAUNCH();
            launch_pdl(pr_wide_scan_kernel<5>, dim3((unsigned)(2 * B)), dim3(1024), 0, st, w.ghist);
            PTK_CHECK_LAUNCH();
            launch_pdl(pr_wide_hist_scatter_kernel<5, true>, sgrid, dim3(PRW_THREADS), 0, st, x, y, iP1, iP2, lx, ly,
                       (const PrWide *)w.wide, w.ghist, w.soa_x, w.soa_y, w.stage_x, w.stage_y, w.bad);
        } else {
            launch_pdl(pr_wide_hist_scatter_kernel<4, false>, sgrid, dim3(PRW_THREADS), 0, st, x, y, iP1, iP2, lx, ly,
                       (const PrWide *)w.wide, w.ghist, w.soa_x, w.soa_y, w.stage_x, w.stage_y, w.bad);
            PTK_CHECK_LAUNCH();
            launch_pdl(pr_wide_scan_kernel<4>, dim3((unsigned)(2 * B)), dim3(1024), 0, st, w.ghist);
            PTK_CHECK_LAUNCH();
            launch_pdl(pr_wide_hist_scatter_kernel<4, true>, sgrid, dim3(PRW_THREADS), 0, st, x, y, iP1, iP2, lx, ly,
                       (const PrWide *)w.wide, w.ghist, w.soa_x, w.soa_y, w.stage_x, w.stage_y, w.bad);
        }
        PTK_CHECK_LAUNCH();
        launch_pdl(pr_wide_leaf_kernel, dim3((unsigned)ceil_div((int64_t)soa_padded((int)Pm) / PR_CHUNK, (int64_t)16), (unsigned)(2 * B)),
                   dim3(256), 0, st, iP1, iP2, lx, ly, (const float4 *)w.stage_x, (const float4 *)w.stage_y, w.soa_x, w.soa_y, w.box_x,
                   w.box_y);
        PTK_CHECK_LAUNCH();
        launch_pdl(pr_wide_inner_kernel, dim3((unsigned)(2 * B)), dim3(1024), 0, st, iP1, iP2, w.box_x, w.box_y);
    } else if (fine) {
        int dev = 0;
        PTK_CHECK_CUDA(cudaGetDevice(&dev));
        if (dev >= 64 || !((g_pr_optin >> dev) & 1ull)) {
            PTK_CHECK_CUDA(cudaFuncSetAttribute(chamfer_pruned_sort_kernel<5>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                                4 * 32768));
            if (dev < 64) g_pr_optin |= 1ull << dev;
        }
        launch_pdl(chamfer_pruned_sort_kernel<5>, dim3((unsigned)(2 * B)), dim3(PR_SORT_THREADS), 4 * 32768, st, x, y, iP1,
                   iP2, lx, ly, w.soa_x, w.soa_y, w.stage_x, w.stage_y, w.box_x, w.box_y, w.bad, w.count, 0);
    } else {
        // <= 32768 points: 16 KB histogram + up to 64 KB of 16-bit cell ranks (the 48 KB default limit covers 16k points)
        const size_t smem = 4 * 4096 + 2 * (size_t)((P1 > P2 ? P1 : P2) + 8);
        int keep = smem <= 48 * 1024 ? 1 : 0;
        launch_pdl(chamfer_pruned_sort_kernel<4>, dim3((unsigned)(2 * B)), dim3(PR_SORT_THREADS), keep ? smem : 4 * 4096, st, x,
                   y, iP1, iP2, lx, ly, w.soa_x, w.soa_y, w.stage_x, w.stage_y, w.box_x, w.box_y, w.bad, w.count, keep);
    }
    PTK_CHECK_LAUNCH();
    u64 *keys_x = dir_only == 1 ? nullptr : w.keys_x;
    u64 *keys_y = dir_only == 0 ? nullptr : w.keys_y;
    // One query per lane.  Two per lane (R = 2) halve the leaf loads per query -- the kernel is bound by the L1 return
    // path -- but the wider query box costs as many extra scans and 72 registers: measured 891 vs 870 us at 256 x 10k,
    // 422 vs 413 us at 16 x 50k.  Kept selectable for development (PTK_PR_R=2, read per call).
    int R = 1;
    if (getenv("PTK_PR_R")) R = atoi(getenv("PTK_PR_R")) == 2 ? 2 : 1;
    dim3 qgrid((unsigned)ceil_div(Pq, (int64_t)PR_QUERY_WARPS * 32 * R), (unsigned)(B * ndir));
    if (R == 2)
        launch_pdl(chamfer_pruned_query_kernel<2>, qgrid, dim3(PR_QUERY_WARPS * 32), 0, st, (const float *)w.soa_x,
                   (const float *)w.soa_y, (const PrBox *)w.box_x, (const PrBox *)w.box_y, (const int *)w.bad, iP1, iP2, lx, ly, keys_x,
                   keys_y, dir_only, w.rescue_x, w.rescue_y, w.count);
    else
        launch_pdl(chamfer_pruned_query_kernel<1>, qgrid, dim3(PR_QUERY_WARPS * 32), 0, st, (const float *)w.soa_x,
                   (const float *)w.soa_y, (const PrBox *)w.box_x, (const PrBox *)w.box_y, (const int *)w.bad, iP1, iP2, lx, ly, keys_x,
                   keys_y, dir_only, w.rescue_x, w.rescue_y, w.count);
    PTK_CHECK_LAUNCH();
    const NNPlan p = plan_nn(B, Pq, Pt, ndir, CH_MINB, CH_CHUNK);
    dim3 rgrid((unsigned)ceil_div(Pq, (int64_t)CH_THREADS * 8), (unsigned)p.n_split, (unsigned)(B * ndir));
    launch_pdl(chamfer_nn_exact2_kernel<8, CH_CHUNK, CH_THREADS, CH_MINB>, rgrid, dim3(CH_THREADS), 0, st, x, y, iP1, iP2,
               lx, ly, p.split_len, p.n_split, w.keys_x, w.keys_y, dir_only, w.rescue_x, w.rescue_y, w.count);
    PTK_CHECK_LAUNCH();
    return PTK_OK;
}

// PTK_CHAMFER_AUTO: the pruned scan pays for its sort once the clouds are large enough (measured crossover,
// tools/chamfer_sweep.py); larger than one top-level group of boxes falls back to the filter scan.
static int resolve_algo(int64_t P1, int64_t P2) {
    int algo = g_chamfer_algo.load(std::memory_order_relaxed);
    const int64_t Pmax = P1 > P2 ? P1 : P2, Pmin = P1 > P2 ? P2 : P1;
    if (algo == PTK_CHAMFER_AUTO) algo = (Pmin >= PTK_CHAMFER_AUTO_MIN_POINTS) ? PTK_CHAMFER_PRUNED : PTK_CHAMFER_FILTER;
    if (algo == PTK_CHAMFER_PRUNED && Pmax > PR_MAX_POINTS) algo = PTK_CHAMFER_FILTER;
    return algo;
}

// lx / ly: per-pair lengths (NULL: every cloud is full).  Plans, grids and the choice of the scan come from the padded
// sizes; the kernels bound their queries and targets by the lengths.
static int launch_nn(const float *x, const float *y, const int64_t *lx, const int64_t *ly, int64_t B, int64_t P1,
                     int64_t P2, const ChamferWs &w, int dir_only, cudaStream_t st) {
    const int algo = resolve_algo(P1, P2);
    if (algo == PTK_CHAMFER_PRUNED) return launch_nn_pruned(x, y, lx, ly, B, P1, P2, w, dir_only, st);
    const int ndir = dir_only >= 0 ? 1 : 2;
    const int64_t Pq = dir_only == 0 ? P1 : (dir_only == 1 ? P2 : (P1 > P2 ? P1 : P2));
    const int64_t Pt = dir_only == 0 ? P2 : (dir_only == 1 ? P1 : (P1 > P2 ? P1 : P2));
    const bool filter = algo == PTK_CHAMFER_FILTER;
    // The filter's exact recheck reads each query's recorded chunk with per-thread vector loads, which needs every cloud
    // of the batch 16-byte aligned.  With 4-byte loads a 64-target recheck costs more than the wider chunks save
    // (DESIGN.md K1), so such batches keep 16-target chunks.
    // The recheck is paid once per query and split, so its share grows as the splits shrink: 64-target chunks also
    // need splits of at least CH_WIDE_MIN_SPLIT targets (fitted on tools/chamfer_layout_bench.py and
    // tools/chamfer_sweep.py: +5 % at 10k targets per split, -4 % at 900).
    auto vec_ok = [&](const float *p, int64_t P) { return (reinterpret_cast<uintptr_t>(p) & 15) == 0 && (B == 1 || P % 4 == 0); };
    bool wide = filter && vec_ok(x, P1) && vec_ok(y, P2);
    NNPlan p = plan_nn(B, Pq, Pt, ndir, filter ? CH_MINB_F : CH_MINB, wide ? CH_CHUNK_F : CH_CHUNK);
    if (wide && p.split_len < CH_WIDE_MIN_SPLIT) {
        wide = false;
        p = plan_nn(B, Pq, Pt, ndir, CH_MINB_F, CH_CHUNK);
    }
    u64 *keys_x = dir_only == 1 ? nullptr : w.keys_x;
    u64 *keys_y = dir_only == 0 ? nullptr : w.keys_y;
    if (p.n_split > 1 && !filter) {  // (the filter path initialises keys and flags in chamfer_prep_kernel)
        if (keys_x) PTK_CHECK_CUDA(cudaMemsetAsync(keys_x, 0xff, sizeof(u64) * B * P1, st));
        if (keys_y) PTK_CHECK_CUDA(cudaMemsetAsync(keys_y, 0xff, sizeof(u64) * B * P2, st));
    }
    dim3 grid((unsigned)ceil_div(Pq, (int64_t)CH_THREADS * p.R), (unsigned)p.n_split,
              (unsigned)(B * ndir));
    PTK_REQUIRE(grid.z <= 65535 && grid.y <= 65535, PTK_ERR_SHAPE,
                "chamfer: batch %lld too large for one launch (max 32767 clouds)", (long long)B);
    const int iP1 = (int)P1, iP2 = (int)P2;
    if (filter) {
        launch_pdl(chamfer_bounds_kernel, dim3((unsigned)B), dim3(1024), 0, st, x, y, iP1, iP2, lx, ly, w.aux, w.count);
        PTK_CHECK_LAUNCH();
        const int Pp = soa_padded(iP1 > iP2 ? iP1 : iP2);
        launch_pdl(chamfer_prep_kernel, dim3((unsigned)ceil_div(Pp, 256), (unsigned)(2 * B)), dim3(256), 0, st, x, y, iP1, iP2,
                   lx, ly, w.aux, w.soa_x, w.soa_y, keys_x, keys_y, w.flag_x, w.flag_y, p.n_split > 1 ? 1 : 0);
        PTK_CHECK_LAUNCH();
#define PTK_FILTER(RR, CC)                                                                                      \
    launch_pdl(chamfer_nn_filter_tma_kernel<RR, CC, CH_THREADS, CH_MINB_F, CH_TT_F>, grid, dim3(CH_THREADS), 0, st,      \
               x, y, iP1, iP2, lx, ly, p.split_len, p.n_split, w.aux, w.soa_x, w.soa_y, w.keys_x, w.keys_y, dir_only, w.rescue_x, \
               w.rescue_y, w.count, w.flag_x, w.flag_y)
        switch (p.R) {
            case 8: if (wide) PTK_FILTER(8, CH_CHUNK_F); else PTK_FILTER(8, CH_CHUNK); break;
            case 4: if (wide) PTK_FILTER(4, CH_CHUNK_F); else PTK_FILTER(4, CH_CHUNK); break;
            default: if (wide) PTK_FILTER(2, CH_CHUNK_F); else PTK_FILTER(2, CH_CHUNK); break;
        }
#undef PTK_FILTER
        PTK_CHECK_LAUNCH();
        // rescue pass over the queued (ambiguous) queries; CTAs beyond the list length exit at once
        dim3 rgrid((unsigned)ceil_div(Pq, (int64_t)CH_THREADS * 8), (unsigned)p.n_split, (unsigned)(B * ndir));
        launch_pdl(chamfer_nn_exact2_kernel<8, CH_CHUNK, CH_THREADS, CH_MINB>, rgrid, dim3(CH_THREADS), 0, st, x, y, iP1, iP2,
                   lx, ly, p.split_len, p.n_split, w.keys_x, w.keys_y, dir_only, w.rescue_x, w.rescue_y, w.count);
        PTK_CHECK_LAUNCH();
        return PTK_OK;
    }
#define PTK_EXACT(RR)                                                                            \
    launch_pdl(chamfer_nn_exact2_kernel<RR, CH_CHUNK, CH_THREADS, CH_MINB>, grid, dim3(CH_THREADS), 0, st, x, y, iP1, iP2, \
               lx, ly, p.split_len, p.n_split, w.keys_x, w.keys_y, dir_only, nullptr, nullptr, nullptr)
    switch (p.R) {
        case 8: PTK_EXACT(8); break;
        case 4: PTK_EXACT(4); break;
        default: PTK_EXACT(2); break;
    }
#undef PTK_EXACT
    PTK_CHECK_LAUNCH();
    return PTK_OK;
}

int chamfer_resolve_algo(int64_t P1, int64_t P2) { return resolve_algo(P1, P2); }  // for the host pipeline (host_api.cu)

}  // namespace ptk

using namespace ptk;

extern "C" size_t ptk_chamfer_workspace_bytes(int64_t B, int64_t P1, int64_t P2) {
    if (B <= 0 || P1 <= 0 || P2 <= 0) return 0;
    return chamfer_ws_bytes(B, P1, P2);
}

extern "C" int ptk_chamfer_set_algo(int algo) {
    PTK_REQUIRE(algo == PTK_CHAMFER_FILTER || algo == PTK_CHAMFER_EXACT || algo == PTK_CHAMFER_PRUNED ||
                    algo == PTK_CHAMFER_AUTO, PTK_ERR_SHAPE,
                "chamfer_set_algo: unknown algorithm %d", algo);
    g_chamfer_algo.store(algo, std::memory_order_relaxed);
    return PTK_OK;
}

#ifdef PTK_PR_STATS
extern "C" int ptk_debug_pr_stats(unsigned long long *out16, int reset) {  // development builds only (not in ptk.h)
    PTK_CHECK_CUDA(cudaDeviceSynchronize());
    PTK_CHECK_CUDA(cudaMemcpyFromSymbol(out16, pr_stats, 128));
    if (reset) {
        unsigned long long z[16] = {0};
        PTK_CHECK_CUDA(cudaMemcpyToSymbol(pr_stats, z, 128));
    }
    return PTK_OK;
}
#endif

extern "C" int ptk_chamfer_get_algo(void) { return g_chamfer_algo.load(std::memory_order_relaxed); }

extern "C" int ptk_chamfer_rescued(const void *workspace, int64_t B, int64_t P1, int64_t P2,
                                   int64_t *n_rescued, ptk_stream_t stream) {
    PTK_REQUIRE(workspace && n_rescued && B > 0 && P1 > 0 && P2 > 0, PTK_ERR_SHAPE, "chamfer_rescued: bad argument");
    const ChamferWs w = carve(const_cast<void *>(workspace), B, P1, P2);
    cudaStream_t st = as_stream(stream);
    unsigned int *h = nullptr;
    PTK_CHECK_CUDA(cudaMallocHost(&h, sizeof(unsigned int) * 2 * B));
    cudaError_t e = cudaMemcpyAsync(h, w.count, sizeof(unsigned int) * 2 * B, cudaMemcpyDeviceToHost, st);
    if (e == cudaSuccess) e = cudaStreamSynchronize(st);
    int64_t n = 0;
    if (e == cudaSuccess)
        for (int64_t i = 0; i < 2 * B; ++i) n += h[i];
    cudaFreeHost(h);
    PTK_CHECK_CUDA(e);
    *n_rescued = resolve_algo(P1, P2) != PTK_CHAMFER_EXACT ? n : 0;
    return PTK_OK;
}

static int check_clouds(const void *x, const void *y, int64_t B, int64_t P1, int64_t P2) {
    PTK_REQUIRE(x && y, PTK_ERR_SHAPE, "chamfer: null cloud pointer");
    PTK_REQUIRE(B > 0 && P1 > 0 && P2 > 0, PTK_ERR_SHAPE,
                "chamfer: empty input (B=%lld, P1=%lld, P2=%lld); point clouds must be non-empty",
                (long long)B, (long long)P1, (long long)P2);
    PTK_REQUIRE(P1 < (1LL << 31) / 3 && P2 < (1LL << 31) / 3, PTK_ERR_SHAPE,
                "chamfer: cloud too large for 32-bit indexing");
    return PTK_OK;
}

static int knn1_fwd(const float *p1, const float *p2, const int64_t *len1, const int64_t *len2, int64_t B, int64_t P1,
                    int64_t P2, float *dist, int32_t *idx, void *workspace, size_t workspace_bytes, ptk_stream_t stream) {
    int rc = check_clouds(p1, p2, B, P1, P2);
    if (rc) return rc;
    PTK_REQUIRE(workspace && workspace_bytes >= chamfer_ws_bytes(B, P1, P2), PTK_ERR_WORKSPACE,
                "knn1: workspace too small (%zu < %zu)", workspace_bytes, chamfer_ws_bytes(B, P1, P2));
    PTK_REQUIRE((reinterpret_cast<uintptr_t>(workspace) & 15) == 0, PTK_ERR_ALIGN, "knn1: workspace must be 16-byte aligned");
    cudaStream_t st = as_stream(stream);
    const ChamferWs w = carve(workspace, B, P1, P2);
    rc = launch_nn(p1, p2, len1, len2, B, P1, P2, w, 0, st);
    if (rc) return rc;
    launch_pdl(chamfer_finalize_kernel, dim3((unsigned)B, (unsigned)fin_splits(P1, P2)), dim3(512), 0, st, w.keys_x, nullptr,
               (int)P1, (int)P2, len1, len2, 1, dist, idx, nullptr, nullptr, nullptr, nullptr);
    PTK_CHECK_LAUNCH();
    return PTK_OK;
}

extern "C" int ptk_knn1_fwd(const float *p1, const float *p2, int64_t B, int64_t P1, int64_t P2,
                            float *dist, int32_t *idx, void *workspace, size_t workspace_bytes,
                            ptk_stream_t stream) {
    PTK_NVTX("ptk_knn1_fwd");
    return knn1_fwd(p1, p2, nullptr, nullptr, B, P1, P2, dist, idx, workspace, workspace_bytes, stream);
}

extern "C" int ptk_knn1_fwd_lengths(const float *p1, const float *p2, const int64_t *len1, const int64_t *len2, int64_t B,
                                    int64_t P1, int64_t P2, float *dist, int32_t *idx, void *workspace,
                                    size_t workspace_bytes, ptk_stream_t stream) {
    PTK_NVTX("ptk_knn1_fwd_lengths");
    return knn1_fwd(p1, p2, len1, len2, B, P1, P2, dist, idx, workspace, workspace_bytes, stream);
}

static int check_reduction(int reduction) {
    PTK_REQUIRE(reduction == PTK_REDUCE_MEAN || reduction == PTK_REDUCE_SUM, PTK_ERR_SHAPE,
                "chamfer: unknown point reduction %d", reduction);
    return PTK_OK;
}

static int chamfer_fwd(const float *x, const float *y, const int64_t *len_x, const int64_t *len_y, int64_t B, int64_t P1,
                       int64_t P2, int reduction, float *dist_x, int32_t *idx_x, float *dist_y, int32_t *idx_y, float *cham,
                       void *workspace, size_t workspace_bytes, ptk_stream_t stream) {
    int rc = check_clouds(x, y, B, P1, P2);
    if (rc) return rc;
    rc = check_reduction(reduction);
    if (rc) return rc;
    PTK_REQUIRE(idx_x && idx_y && cham, PTK_ERR_SHAPE, "chamfer_fwd: idx_x, idx_y and cham are required");
    PTK_REQUIRE(workspace && workspace_bytes >= ptk_chamfer_workspace_bytes(B, P1, P2),
                PTK_ERR_WORKSPACE, "chamfer_fwd: workspace too small (%zu < %zu)", workspace_bytes,
                ptk_chamfer_workspace_bytes(B, P1, P2));
    PTK_REQUIRE((reinterpret_cast<uintptr_t>(workspace) & 15) == 0, PTK_ERR_ALIGN,
                "chamfer_fwd: workspace must be 16-byte aligned");
    cudaStream_t st = as_stream(stream);
    const ChamferWs w = carve(workspace, B, P1, P2);
    rc = launch_nn(x, y, len_x, len_y, B, P1, P2, w, -1, st);
    if (rc) return rc;
    const int nsp = fin_splits(P1, P2);
    const int mean = reduction == PTK_REDUCE_MEAN ? 1 : 0;
    // partial sums of the slices: the rescue flags are dead once the scan is over (flag_x holds B * P1 >= 2 * B * nsp words)
    float *partial = reinterpret_cast<float *>(w.flag_x);
    launch_pdl(chamfer_finalize_kernel, dim3((unsigned)B, (unsigned)nsp), dim3(512), 0, st, w.keys_x, w.keys_y, (int)P1, (int)P2,
               len_x, len_y, mean, dist_x, idx_x, dist_y, idx_y, cham, partial);
    if (nsp > 1) {
        PTK_CHECK_LAUNCH();
        launch_pdl(chamfer_finalize_sum_kernel, dim3((unsigned)ceil_div(B, (int64_t)128)), dim3(128), 0, st, (const float *)partial,
                   (int)B, nsp, (int)P1, (int)P2, len_x, len_y, mean, cham);
    }
    PTK_CHECK_LAUNCH();
    return PTK_OK;
}

extern "C" int ptk_chamfer_fwd(const float *x, const float *y, int64_t B, int64_t P1, int64_t P2,
                               float *dist_x, int32_t *idx_x, float *dist_y, int32_t *idx_y,
                               float *cham, void *workspace, size_t workspace_bytes,
                               ptk_stream_t stream) {
    PTK_NVTX("ptk_chamfer_fwd");
    return chamfer_fwd(x, y, nullptr, nullptr, B, P1, P2, PTK_REDUCE_MEAN, dist_x, idx_x, dist_y, idx_y, cham, workspace,
                       workspace_bytes, stream);
}

extern "C" int ptk_chamfer_fwd_lengths(const float *x, const float *y, const int64_t *len_x, const int64_t *len_y, int64_t B,
                                       int64_t P1, int64_t P2, int reduction, float *dist_x, int32_t *idx_x, float *dist_y,
                                       int32_t *idx_y, float *cham, void *workspace, size_t workspace_bytes,
                                       ptk_stream_t stream) {
    PTK_NVTX("ptk_chamfer_fwd_lengths");
    return chamfer_fwd(x, y, len_x, len_y, B, P1, P2, reduction, dist_x, idx_x, dist_y, idx_y, cham, workspace,
                       workspace_bytes, stream);
}

static int chamfer_bwd(const float *x, const float *y, const int64_t *len_x, const int64_t *len_y, const int32_t *idx_x,
                       const int32_t *idx_y, const float *grad_cham, int64_t B, int64_t P1, int64_t P2, int reduction,
                       float *grad_x, float *grad_y, ptk_stream_t stream) {
    int rc = check_clouds(x, y, B, P1, P2);
    if (rc) return rc;
    rc = check_reduction(reduction);
    if (rc) return rc;
    PTK_REQUIRE(idx_x && idx_y && grad_cham, PTK_ERR_SHAPE, "chamfer_bwd: null index / grad pointer");
    if (!grad_x && !grad_y) return PTK_OK;
    cudaStream_t st = as_stream(stream);
    const int64_t Pm = P1 > P2 ? P1 : P2;
    dim3 grid((unsigned)ceil_div(Pm, 256), (unsigned)B);
    PTK_REQUIRE(B <= 65535, PTK_ERR_SHAPE, "chamfer_bwd: batch too large");
    const int mean = reduction == PTK_REDUCE_MEAN ? 1 : 0;
    launch_pdl(chamfer_bwd_direct_kernel, grid, dim3(256), 0, st, x, y, idx_x, idx_y, grad_cham, (int)P1, (int)P2, len_x, len_y,
               mean, grad_x, grad_y);
    PTK_CHECK_LAUNCH();
    launch_pdl(chamfer_bwd_scatter_kernel, grid, dim3(256), 0, st, x, y, idx_x, idx_y, grad_cham, (int)P1, (int)P2, len_x, len_y,
               mean, grad_x, grad_y);
    PTK_CHECK_LAUNCH();
    return PTK_OK;
}

extern "C" int ptk_chamfer_bwd(const float *x, const float *y, const int32_t *idx_x,
                               const int32_t *idx_y, const float *grad_cham, int64_t B, int64_t P1,
                               int64_t P2, float *grad_x, float *grad_y, ptk_stream_t stream) {
    PTK_NVTX("ptk_chamfer_bwd");
    return chamfer_bwd(x, y, nullptr, nullptr, idx_x, idx_y, grad_cham, B, P1, P2, PTK_REDUCE_MEAN, grad_x, grad_y, stream);
}

extern "C" int ptk_chamfer_bwd_lengths(const float *x, const float *y, const int64_t *len_x, const int64_t *len_y,
                                       const int32_t *idx_x, const int32_t *idx_y, const float *grad_cham, int64_t B,
                                       int64_t P1, int64_t P2, int reduction, float *grad_x, float *grad_y,
                                       ptk_stream_t stream) {
    PTK_NVTX("ptk_chamfer_bwd_lengths");
    return chamfer_bwd(x, y, len_x, len_y, idx_x, idx_y, grad_cham, B, P1, P2, reduction, grad_x, grad_y, stream);
}
