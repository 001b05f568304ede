/*
 * tests/f64_reference.c -- TEST INFRASTRUCTURE (double-precision reference of the discrete scheme), not product code.
 *
 * The engine's estimators restated in double, path by path, so that a test can look at single antithetic pairs.  It
 * shares with the float oracle (oracle/hw1f_oracle.c) only what defines WHICH normals a path sees:
 *   - the XORWOW integer stream (xw_init / xw_next of oracle/xorwow_ref.c, bit-exact against cuRAND);
 *   - cuRAND's two float uniforms of Box-Muller, u = x 2^-32 + 2^-33 and v = y 2pi 2^-32 + pi 2^-32 (one fused
 *     multiply-add each, curand_normal.h), which are exact float values and define the pair's normals.
 * Everything after that is double: the radius sqrt(-2 ln u), sin v and cos v (libm), and the recursion of both
 * antithetic twins,
 *     r_{i+1} = r_i e + d_i +/- sig_st G_i,     I_{i+1} = I_i + (r_i + r_{i+1}) dt / 2      (r_0 given, I_0 = 0).
 * The drift table d_i, the step constants and the payoffs are built by tests/f64_reference.py (float64 numpy) from
 * the model's parameters; this file only walks the paths, because that is where the time goes.
 *
 * Offsets follow curand_normal(): normal 2k is the sin half of the k-th Box-Muller pair of the subsequence, normal 2k + 1
 * its cos half; a path that starts at an odd offset begins with the cos half of pair offset / 2.
 *
 * Built by tests/f64_reference.py with the flags of oracle/Makefile into the temporary directory.
 */
#include <math.h>
#include <stdint.h>
#include <stdlib.h>
#include <string.h>

#include "xorwow_ref.h"

static inline float as_float(uint32_t u)
{
    float f;
    memcpy(&f, &u, 4);
    return f;
}

/* the pair (sin half, cos half) of one Box-Muller draw, in double from curand's float uniforms */
static inline void box_muller_f64(uint32_t x, uint32_t y, double* n_sin, double* n_cos)
{
    const float u = fmaf((float)x, as_float(0x2f800000u), as_float(0x2f000000u));
    const float v = fmaf((float)y, as_float(0x30c90fdbu), as_float(0x30490fdbu));
    const double s = sqrt(-2.0 * log((double)u));
    *n_sin = s * sin((double)v);
    *n_cos = s * cos((double)v);
}

/* normals [offset, offset + n) of one subsequence */
static void normals_f64(uint64_t seed, uint64_t subsequence, uint64_t offset, int n, double* out)
{
    xw_state st;
    xw_init(seed, subsequence, 2 * (offset / 2), &st);
    int k = 0;
    if (offset & 1) {
        double a, b;
        const uint32_t x = xw_next(&st), y = xw_next(&st);
        box_muller_f64(x, y, &a, &b);
        if (n > 0) out[k++] = b;
    }
    while (k < n) {
        double a, b;
        const uint32_t x = xw_next(&st), y = xw_next(&st);
        box_muller_f64(x, y, &a, &b);
        out[k++] = a;
        if (k < n) out[k++] = b;
    }
}

void f64_normals(uint64_t seed, uint64_t subsequence, uint64_t offset, int n, double* out)
{
    xw_build_tables();
    normals_f64(seed, subsequence, offset, n, out);
}

/*
 * For pairs q = 0 .. n_pairs-1 (subsequence first_path + q, normals from `offset`), walk both twins through
 * eval_steps[n_eval - 1] steps and store, at every step k = eval_steps[j] (non-decreasing, >= 0),
 *     out[(q n_eval + j) 4 + {0, 1, 2, 3}] = {r(+G), r(-G), I(+G), I(-G)} after k steps.
 * drift[n_steps_table] (>= the last eval step), e = e^{-a dt}, dt, sig_st and r0 as the caller's model defines them.
 */
void f64_pair_states(const double* drift, double e, double dt, double sig_st, double r0, uint64_t seed,
                     uint64_t first_path, int64_t n_pairs, uint64_t offset, const int* eval_steps, int n_eval,
                     double* out)
{
    xw_build_tables();
    const int n_last = n_eval > 0 ? eval_steps[n_eval - 1] : 0;
#pragma omp parallel
    {
        double* G = (double*)malloc((size_t)(n_last > 0 ? n_last : 1) * sizeof(double));
#pragma omp for schedule(static)
        for (int64_t q = 0; q < n_pairs; q++) {
            normals_f64(seed, first_path + (uint64_t)q, offset, n_last, G);
            double r1 = r0, r2 = r0, I1 = 0.0, I2 = 0.0;
            int step = 0;
            for (int j = 0; j < n_eval; j++) {
                for (; step < eval_steps[j]; step++) {
                    const double n1 = r1 * e + drift[step] + sig_st * G[step];
                    const double n2 = r2 * e + drift[step] - sig_st * G[step];
                    I1 += 0.5 * (r1 + n1) * dt;
                    I2 += 0.5 * (r2 + n2) * dt;
                    r1 = n1;
                    r2 = n2;
                }
                double* o = out + ((size_t)q * n_eval + j) * 4;
                o[0] = r1; o[1] = r2; o[2] = I1; o[3] = I2;
            }
        }
        free(G);
    }
}
