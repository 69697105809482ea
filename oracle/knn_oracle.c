/* CPU oracle of ptk_knn_fwd_lengths (test infrastructure; built by knn_oracle.py).
 * K nearest neighbours of homogeneous clouds with the selection rule of PyTorch3D's knn_cpu.cpp:
 * K slots of (+inf, 0); j ascending; (d, j) enters when d < slot[K-1].d (strict: NaN and +inf never
 * enter, an equal distance never displaces a lower index) and is inserted after every slot whose
 * distance is <= d.  dist / idx are (B,P1,K); slots k >= P2 are (0, 0), as PyTorch3D pads them.
 * d is sqdist3 of ptk_oracle.c: fma(dz,dz, fma(dy,dy, dx*dx)), or (dx*dx + dy*dy) + dz*dz. */
#include <math.h>
#include <stdint.h>

static inline float sqdist3(const float *a, const float *b, int use_fma) {
    float dx = a[0] - b[0];
    float dy = a[1] - b[1];
    float dz = a[2] - b[2];
    float d = dx * dx;
    if (use_fma) {
        d = fmaf(dy, dy, d);
        d = fmaf(dz, dz, d);
    } else {
        d = d + dy * dy;
        d = d + dz * dz;
    }
    return d;
}

void orc_knn(const float *p1, const float *p2, int64_t B, int64_t P1, int64_t P2, int64_t K,
             float *dist, int32_t *idx, int use_fma) {
#pragma omp parallel for collapse(2) schedule(static)
    for (int64_t b = 0; b < B; ++b) {
        for (int64_t i = 0; i < P1; ++i) {
            const float *q = p1 + (b * P1 + i) * 3;
            const float *t = p2 + b * P2 * 3;
            float *sd = dist + (b * P1 + i) * K;
            int32_t *si = idx + (b * P1 + i) * K;
            for (int64_t k = 0; k < K; ++k) {
                sd[k] = INFINITY;
                si[k] = 0;
            }
            for (int64_t j = 0; j < P2; ++j) {
                float d = sqdist3(q, t + j * 3, use_fma);
                if (!(d < sd[K - 1])) continue;
                int64_t k = K - 1;
                while (k > 0 && sd[k - 1] > d) {
                    sd[k] = sd[k - 1];
                    si[k] = si[k - 1];
                    --k;
                }
                sd[k] = d;
                si[k] = (int32_t)j;
            }
            for (int64_t k = P2; k < K; ++k) {
                sd[k] = 0.0f;
                si[k] = 0;
            }
        }
    }
}
