/*
 * tests/gw_assign_oracle.c -- TEST INFRASTRUCTURE ONLY: the pinned-order GW assignment that defines the integer result of
 * gfs_gw_project / gfs_gw_project_tc (the formula in the header of gfs-3dseg_gws_b200/csrc/rowsel.cu; model/capl.py:344-353).
 * tests/test_gpu_wide_dictionary.py compiles it with the flags of oracle/gfs_oracle.py:build_c into a temporary directory.
 *
 *   dot(a, b)  = fma chain over channels c = 0..D-1 ascending, starting from +0.0f (the pinned order of oracle/gfs_oracle.c)
 *   score(n,g) = dot(ec_n, gp_g) * (10 / max(sqrt(dot(ec_n, ec_n)), 1e-12))
 *   assignment = argmax_g score, ties -> smaller g
 */
#include <math.h>
#include <stddef.h>
#include <stdint.h>

static inline float dot_chain(const float* a, long sa, const float* b, long sb, int C) {
    float acc = 0.0f;
    for (int c = 0; c < C; ++c) acc = fmaf(a[c * sa], b[c * sb], acc);
    return acc;
}

/* ec (B, D, N) fp32 channel-major, gp (G, D) row-major L2-normalised words -> assignment (B, N) int32 */
int gw_assign_exact(const float* ec, int B, int D, int N, const float* gp, int G, int32_t* assignment) {
#pragma omp parallel for schedule(static) collapse(2)
    for (int b = 0; b < B; ++b)
        for (int n = 0; n < N; ++n) {
            const float* x = ec + (size_t)b * D * N + n;
            const float nrm = dot_chain(x, N, x, N, D);
            const float inv = 10.0f / fmaxf(sqrtf(nrm), 1e-12f);
            float bs = -INFINITY;
            int bg = 0;
            for (int g = 0; g < G; ++g) {
                const float s = dot_chain(x, N, gp + (size_t)g * D, 1, D) * inv;
                if (s > bs) {
                    bs = s;
                    bg = g;
                }
            }
            assignment[(size_t)b * N + n] = bg;
        }
    return 0;
}
