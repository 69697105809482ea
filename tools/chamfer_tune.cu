// Variant sweep for chamfer_nn_kernel (development tool, not part of the library).
//   nvcc -gencode arch=compute_100a,code=sm_100a -O3 -lineinfo -I include -I active-3d-vision-and-touch_b200/csrc \
//        tools/chamfer_tune.cu active-3d-vision-and-touch_b200/csrc/abi.cu -o tools/chamfer_tune
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <vector>

#include "chamfer_kernel2.cuh"

using namespace ptk;

#define CK(x) do { cudaError_t e = (x); if (e != cudaSuccess) { printf("CUDA error %s at %d\n", cudaGetErrorString(e), __LINE__); exit(1); } } while (0)

__device__ float urand(size_t i, unsigned seed) {
    unsigned h = (unsigned)i * 2654435761u ^ seed;
    h ^= h >> 16; h *= 0x85ebca6bu; h ^= h >> 13; h *= 0xc2b2ae35u; h ^= h >> 16;
    return (h >> 8) * (1.0f / 16777216.0f);
}
// mode 0: uniform cube; 1: sphere surface r=0.25; 2: thin rod (config 1 extents); 3: cube, cloud tiled x4 (exact duplicates)
__global__ void fill(float *p, size_t n, unsigned seed, int mode, int P) {
    size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x;
    if (i >= n) return;
    size_t pt = i / 3; int c = (int)(i % 3);
    if (mode == 3) { size_t b = pt / P, j = pt % P; pt = b * P + j % (P / 4); }
    float u = urand(pt * 3 + c, seed);
    if (mode == 0 || mode == 3) p[i] = u - 0.5f;
    if (mode == 2) p[i] = u * (c == 0 ? 0.004f : (c == 1 ? 0.0107f : 0.192f));
    if (mode == 1) {
        float z = 2.f * urand(pt * 3, seed) - 1.f, ph = 6.2831853f * urand(pt * 3 + 1, seed), r = sqrtf(fmaxf(0.f, 1.f - z * z));
        p[i] = 0.25f * (c == 0 ? r * cosf(ph) : (c == 1 ? r * sinf(ph) : z));
    }
}

__global__ void checksum(const unsigned long long *k, size_t n, unsigned long long *out) {
    size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x;
    if (i < n) atomicAdd(out, k[i] * (2 * i + 1));
}

template <int R, int CHUNK, int THREADS, int MINB>
float run(const char *name, const float *x, const float *y, int B, int P, unsigned long long *kx,
          unsigned long long *ky, unsigned long long *d_sum, unsigned long long ref, int reps) {
    dim3 grid((P + THREADS * R - 1) / (THREADS * R), 1, B * 2);
    int split_len = ((P + CHUNK - 1) / CHUNK) * CHUNK;
    cudaEvent_t a, b;
    CK(cudaEventCreate(&a)); CK(cudaEventCreate(&b));
    for (int i = 0; i < 2; ++i)
        chamfer_nn_kernel<R, CHUNK, THREADS, MINB><<<grid, THREADS>>>(x, y, P, P, split_len, 1, kx, ky, -1);
    CK(cudaDeviceSynchronize());
    CK(cudaEventRecord(a));
    for (int i = 0; i < reps; ++i)
        chamfer_nn_kernel<R, CHUNK, THREADS, MINB><<<grid, THREADS>>>(x, y, P, P, split_len, 1, kx, ky, -1);
    CK(cudaEventRecord(b));
    CK(cudaDeviceSynchronize());
    float ms;
    CK(cudaEventElapsedTime(&ms, a, b));
    ms /= reps;
    CK(cudaMemset(d_sum, 0, 8));
    size_t n = (size_t)B * P;
    checksum<<<(unsigned)((n + 255) / 256), 256>>>(kx, n, d_sum);
    checksum<<<(unsigned)((n + 255) / 256), 256>>>(ky, n, d_sum);
    unsigned long long h;
    CK(cudaMemcpy(&h, d_sum, 8, cudaMemcpyDeviceToHost));
    cudaFuncAttributes fa;
    CK(cudaFuncGetAttributes(&fa, chamfer_nn_kernel<R, CHUNK, THREADS, MINB>));
    int occ = 0;
    CK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, chamfer_nn_kernel<R, CHUNK, THREADS, MINB>, THREADS, 0));
    double evals = 2.0 * B * (double)P * P;
    double peak = 128.0 * 148 * 1.965e9 / 6.0;
    printf("%-28s R=%d chunk=%2d thr=%3d minb=%d regs=%3d occ=%d ctas=%5u  %8.3f ms  %6.3f Tevals/s  frac=%.3f  %s\n", name, R,
           CHUNK, THREADS, MINB, fa.numRegs, occ, grid.x * grid.z, ms, evals / ms / 1e9, evals / (ms * 1e-3) / peak,
           ref == 0 ? "(ref)" : (h == ref ? "OK" : "MISMATCH"));
    fflush(stdout);
    return ref == 0 ? (float)0 : ms;
}

template <int R, int CHUNK, int THREADS, int MINB>
void run_exact2(const char *name, const float *x, const float *y, int B, int P, unsigned long long *kx,
                unsigned long long *ky, unsigned long long *d_sum, unsigned long long ref, int reps) {
    dim3 grid((P + THREADS * R - 1) / (THREADS * R), 1, B * 2);
    int split_len = ((P + CHUNK - 1) / CHUNK) * CHUNK;
    cudaEvent_t a, b;
    CK(cudaEventCreate(&a)); CK(cudaEventCreate(&b));
    auto launch = [&]() { chamfer_nn_exact2_kernel<R, CHUNK, THREADS, MINB><<<grid, THREADS>>>(x, y, P, P, nullptr, nullptr, split_len, 1, kx, ky, -1, nullptr, nullptr, nullptr); };
    launch(); launch();
    CK(cudaDeviceSynchronize());
    CK(cudaEventRecord(a));
    for (int i = 0; i < reps; ++i) launch();
    CK(cudaEventRecord(b));
    CK(cudaDeviceSynchronize());
    float ms;
    CK(cudaEventElapsedTime(&ms, a, b));
    ms /= reps;
    CK(cudaMemset(d_sum, 0, 8));
    size_t n = (size_t)B * P;
    checksum<<<(unsigned)((n + 255) / 256), 256>>>(kx, n, d_sum);
    checksum<<<(unsigned)((n + 255) / 256), 256>>>(ky, n, d_sum);
    unsigned long long h;
    CK(cudaMemcpy(&h, d_sum, 8, cudaMemcpyDeviceToHost));
    cudaFuncAttributes fa;
    CK(cudaFuncGetAttributes(&fa, chamfer_nn_exact2_kernel<R, CHUNK, THREADS, MINB>));
    double evals = 2.0 * B * (double)P * P;
    double peak = 128.0 * 148 * 1.965e9 / 6.0;
    printf("exact2 %-21s R=%d chunk=%2d thr=%3d minb=%d regs=%3d ctas=%5u  %8.3f ms  %6.3f Tevals/s  frac6=%.3f  %s\n", name, R,
           CHUNK, THREADS, MINB, fa.numRegs, grid.x * grid.z, ms, evals / ms / 1e9, evals / (ms * 1e-3) / peak,
           h == ref ? "OK" : "MISMATCH");
    fflush(stdout);
}

template <int R, int CHUNK, int THREADS, int MINB, int TT, bool PK>
void run_filter(const char *name, const float *x, const float *y, int B, int P, unsigned long long *kx,
                unsigned long long *ky, unsigned long long *d_sum, unsigned long long ref, int reps, PairAux *aux,
                unsigned int *d_amb) {
    dim3 grid((P + THREADS * R - 1) / (THREADS * R), 1, B * 2);
    int split_len = ((P + CHUNK - 1) / CHUNK) * CHUNK;
    cudaEvent_t a, b;
    CK(cudaEventCreate(&a)); CK(cudaEventCreate(&b));
    static int *rescue = nullptr;
    static unsigned int *rcount = nullptr;
    if (!rescue) { CK(cudaMalloc(&rescue, 8 * (size_t)B * P)); CK(cudaMalloc(&rcount, 8 * (size_t)B)); }
    dim3 rgrid((P + 128 * 8 - 1) / (128 * 8), 1, B * 2);
    auto launch = [&](unsigned int *) {
        chamfer_bounds_kernel<<<B, 1024>>>(x, y, P, P, nullptr, nullptr, aux, rcount);
        chamfer_nn_filter_kernel<R, CHUNK, THREADS, MINB, TT, PK><<<grid, THREADS>>>(x, y, P, P, split_len, 1, aux, kx, ky, -1, rescue, rescue + (size_t)B * P, rcount, nullptr, nullptr);
        chamfer_nn_exact2_kernel<8, 16, 128, 3><<<rgrid, 128>>>(x, y, P, P, nullptr, nullptr, split_len, 1, kx, ky, -1, rescue, rescue + (size_t)B * P, rcount);
    };
    launch(nullptr);
    CK(cudaDeviceSynchronize());
    unsigned int amb = 0;
    {
        std::vector<unsigned int> hc(2 * B);
        CK(cudaMemcpy(hc.data(), rcount, 8 * (size_t)B, cudaMemcpyDeviceToHost));
        for (auto v : hc) amb += v;
    }
    launch(nullptr);
    CK(cudaDeviceSynchronize());
    CK(cudaEventRecord(a));
    for (int i = 0; i < reps; ++i) launch(nullptr);
    CK(cudaEventRecord(b));
    CK(cudaDeviceSynchronize());
    float ms;
    CK(cudaEventElapsedTime(&ms, a, b));
    ms /= reps;
    CK(cudaMemset(d_sum, 0, 8));
    size_t n = (size_t)B * P;
    checksum<<<(unsigned)((n + 255) / 256), 256>>>(kx, n, d_sum);
    checksum<<<(unsigned)((n + 255) / 256), 256>>>(ky, n, d_sum);
    unsigned long long h;
    CK(cudaMemcpy(&h, d_sum, 8, cudaMemcpyDeviceToHost));
    cudaFuncAttributes fa;
    CK(cudaFuncGetAttributes(&fa, chamfer_nn_filter_kernel<R, CHUNK, THREADS, MINB, TT, PK>));
    double evals = 2.0 * B * (double)P * P;
    double peak = 128.0 * 148 * 1.965e9 / 3.0;
    printf("filter%s %-21s R=%d chunk=%2d thr=%3d minb=%d regs=%3d ctas=%5u  %8.3f ms  %6.3f Tevals/s  frac3=%.3f  amb=%.4f%%  %s\n", PK ? "2" : "1", name, R,
           CHUNK, THREADS, MINB, fa.numRegs, grid.x * grid.z, ms, evals / ms / 1e9, evals / (ms * 1e-3) / peak,
           100.0 * amb / (2.0 * n), h == ref ? "OK" : "MISMATCH");
    fflush(stdout);
}

template <int R, int CHUNK, int THREADS, int MINB, int TT>
void run_tma(const char *name, const float *x, const float *y, int B, int P, unsigned long long *kx,
             unsigned long long *ky, unsigned long long *d_sum, unsigned long long ref, int reps, PairAux *aux) {
    dim3 grid((P + THREADS * R - 1) / (THREADS * R), 1, B * 2);
    int split_len = ((P + CHUNK - 1) / CHUNK) * CHUNK;
    cudaEvent_t a, b;
    CK(cudaEventCreate(&a)); CK(cudaEventCreate(&b));
    static int *rescue = nullptr;
    static unsigned int *rcount = nullptr;
    static float *soa = nullptr;
    const int Pp = soa_padded(P);
    if (!rescue) { CK(cudaMalloc(&rescue, 8 * (size_t)B * P)); CK(cudaMalloc(&rcount, 8 * (size_t)B)); CK(cudaMalloc(&soa, 32 * (size_t)B * Pp)); }
    float *soa_x = soa, *soa_y = soa + (size_t)B * 4 * Pp;
    dim3 rgrid((P + 128 * 8 - 1) / (128 * 8), 1, B * 2);
    dim3 pgrid((Pp + 255) / 256, 2 * B);
    auto launch = [&]() {
        chamfer_bounds_kernel<<<B, 1024>>>(x, y, P, P, nullptr, nullptr, aux, rcount);
        chamfer_prep_kernel<<<pgrid, 256>>>(x, y, P, P, nullptr, nullptr, aux, soa_x, soa_y, nullptr, nullptr, nullptr, nullptr, 0);
        chamfer_nn_filter_tma_kernel<R, CHUNK, THREADS, MINB, TT><<<grid, THREADS>>>(x, y, P, P, nullptr, nullptr, split_len, 1, aux, soa_x, soa_y, kx, ky, -1, rescue, rescue + (size_t)B * P, rcount, nullptr, nullptr);
        chamfer_nn_exact2_kernel<8, 16, 128, 3><<<rgrid, 128>>>(x, y, P, P, nullptr, nullptr, split_len, 1, kx, ky, -1, rescue, rescue + (size_t)B * P, rcount);
    };
    launch();
    CK(cudaDeviceSynchronize());
    unsigned int amb = 0;
    {
        std::vector<unsigned int> hc(2 * B);
        CK(cudaMemcpy(hc.data(), rcount, 8 * (size_t)B, cudaMemcpyDeviceToHost));
        for (auto v : hc) amb += v;
    }
    launch();
    CK(cudaDeviceSynchronize());
    CK(cudaEventRecord(a));
    for (int i = 0; i < reps; ++i) launch();
    CK(cudaEventRecord(b));
    CK(cudaDeviceSynchronize());
    float ms;
    CK(cudaEventElapsedTime(&ms, a, b));
    ms /= reps;
    CK(cudaMemset(d_sum, 0, 8));
    size_t n = (size_t)B * P;
    checksum<<<(unsigned)((n + 255) / 256), 256>>>(kx, n, d_sum);
    checksum<<<(unsigned)((n + 255) / 256), 256>>>(ky, n, d_sum);
    unsigned long long h;
    CK(cudaMemcpy(&h, d_sum, 8, cudaMemcpyDeviceToHost));
    cudaFuncAttributes fa;
    CK(cudaFuncGetAttributes(&fa, chamfer_nn_filter_tma_kernel<R, CHUNK, THREADS, MINB, TT>));
    double evals = 2.0 * B * (double)P * P;
    double peak = 128.0 * 148 * 1.965e9 / 3.0;
    printf("tma     %-21s R=%d chunk=%2d thr=%3d minb=%d regs=%3d ctas=%5u  %8.3f ms  %6.3f Tevals/s  frac3=%.3f  amb=%.4f%%  %s\n", name, R,
           CHUNK, THREADS, MINB, fa.numRegs, grid.x * grid.z, ms, evals / ms / 1e9, evals / (ms * 1e-3) / peak,
           100.0 * amb / (2.0 * n), h == ref ? "OK" : "MISMATCH");
    fflush(stdout);
}

static const char *g_only = nullptr;
static bool want(const char *name) { return g_only == nullptr || strstr(name, g_only) != nullptr; }

int main(int argc, char **argv) {
    g_only = getenv("TUNE_ONLY");
    int B = argc > 1 ? atoi(argv[1]) : 256, P = argc > 2 ? atoi(argv[2]) : 10000, reps = argc > 3 ? atoi(argv[3]) : 5;
    int mode = argc > 4 ? atoi(argv[4]) : 0;
    printf("data mode %d\n", mode);
    size_t n = (size_t)B * P;
    float *x, *y;
    unsigned long long *kx, *ky, *d_sum;
    CK(cudaMalloc(&x, n * 12)); CK(cudaMalloc(&y, n * 12));
    CK(cudaMalloc(&kx, n * 8)); CK(cudaMalloc(&ky, n * 8)); CK(cudaMalloc(&d_sum, 8));
    fill<<<(unsigned)((n * 3 + 255) / 256), 256>>>(x, n * 3, 1u, mode == 3 ? 0 : mode, P);
    fill<<<(unsigned)((n * 3 + 255) / 256), 256>>>(y, n * 3, 2u, mode, P);
    CK(cudaDeviceSynchronize());
    // reference checksum from the baseline variant
    run<8, 16, 256, 2>("baseline", x, y, B, P, kx, ky, d_sum, 0, 1);
    unsigned long long ref;
    CK(cudaMemcpy(&ref, d_sum, 8, cudaMemcpyDeviceToHost));
#define V(R, C, T, M) if (want("V" #R "," #C "," #T "," #M)) run<R, C, T, M>(#R "," #C "," #T "," #M, x, y, B, P, kx, ky, d_sum, ref, reps)
#define E(R, C, T, M) if (want("E" #R "," #C "," #T "," #M)) run_exact2<R, C, T, M>(#R "," #C "," #T "," #M, x, y, B, P, kx, ky, d_sum, ref, reps)
#define F(R, C, T, M, TT) if (want("F" #R "," #C "," #T "," #M "," #TT)) run_filter<R, C, T, M, TT, true>(#R "," #C "," #T "," #M "," #TT, x, y, B, P, kx, ky, d_sum, ref, reps, aux, d_amb)
#define G(R, C, T, M, TT) if (want("G" #R "," #C "," #T "," #M "," #TT)) run_filter<R, C, T, M, TT, false>(#R "," #C "," #T "," #M "," #TT, x, y, B, P, kx, ky, d_sum, ref, reps, aux, d_amb)
#define T(R, C, T_, M, TT) if (want("T" #R "," #C "," #T_ "," #M "," #TT)) run_tma<R, C, T_, M, TT>(#R "," #C "," #T_ "," #M "," #TT, x, y, B, P, kx, ky, d_sum, ref, reps, aux)
    PairAux *aux;
    unsigned int *d_amb;
    CK(cudaMalloc(&aux, sizeof(PairAux) * B)); CK(cudaMalloc(&d_amb, 4));
    V(8, 16, 128, 3);
    // chunk widths of the TMA filter scan, interleaved so that clock and neighbour drift hit every width alike
    const int rounds = getenv("TUNE_ROUNDS") ? atoi(getenv("TUNE_ROUNDS")) : 1;
    for (int i = 0; i < rounds; ++i) {
        T(8, 16, 128, 4, 1024);
        T(8, 32, 128, 4, 1024);
        T(8, 64, 128, 4, 1024);
    }
    return 0;
}
