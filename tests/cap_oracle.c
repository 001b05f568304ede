/*
 * tests/cap_oracle.c -- TEST INFRASTRUCTURE (CPU oracle of the cap / floor strip), not product code.
 *
 * The strip estimator of hw1f_cap_floor restated on the CPU: the reference-order float sequence of orc_zbc_moments
 * (bond_setup, hw_step, libm in place of MUFU) evaluated at every reset step of each pair of paths.  It is a separate
 * translation unit that includes the oracle's own source, so that it runs the oracle's static RNG, Box-Muller, step and
 * bond-plan code itself instead of a copy of it.  Built by tests/cap_oracle.py with the flags of oracle/Makefile.
 *
 * One caplet = one bond option on (T_reset, T_pay), strike K, multiplier N, read at reset step `step` (non-decreasing
 * along the strip, >= 1); kind 0: cap (puts, N D (K - P)^+), 1: floor (calls, N D (P - K)^+).  mom[5 (n + 1)]: per
 * caplet and then for the strip, sums over antithetic PAIRS of X, Y, X^2, Y^2, XY with X = N (x(+G) + x(-G)),
 * Y = N (D P (+G) + D P (-G)); the strip's X, Y are the sums over the caplets.
 */
#include "hw1f_oracle.c"

typedef struct {
    float T_reset, T_pay, K, N;
    int32_t step, reserved;
} orc_caplet;

/* ---- caps and floors -------------------------------------------------------------- */
void orc_cap_moments(const orc_params* p, float sigma, float sig_st, const float* drift,
                     uint64_t seed, uint64_t first_path, int64_t n_pairs, uint64_t offset_normals,
                     int kind, const orc_caplet* caps, int n, const float* P_mkt, const float* f_mkt, double* mom)
{
    xw_build_tables();
    FTZ_SCOPE_BEGIN
    const float exp_adt = orc_exp_adt(p), dt = orc_dt(p), r0 = p->r0;
    const float sgn = kind == 0 ? -1.0f : 1.0f;
    const int nq = 5 * (n + 1), n_last = caps[n - 1].step;
    bond_consts* bc = (bond_consts*)malloc((size_t)n * sizeof(bond_consts));
    for (int i = 0; i < n; i++) bc[i] = bond_setup(p, sigma, caps[i].T_reset, caps[i].T_pay, P_mkt, f_mkt);
    for (int k = 0; k < nq; k++) mom[k] = 0.0;
#pragma omp parallel
    {
        FTZ_THREAD
        double* loc = (double*)calloc((size_t)nq, sizeof(double));
#pragma omp for schedule(static)
        for (int64_t q = 0; q < n_pairs; q++) {
            normal_stream ns;
            ns_init(&ns, seed, first_path + (uint64_t)q, offset_normals);
            float r1 = r0, r2 = r0, I1 = 0.0f, I2 = 0.0f;
            double Xs = 0.0, Ys = 0.0;
            int step = 0;
            for (int i = 0; i < n; i++) {
                for (; step < caps[i].step && step < n_last; step++) {
                    float d = drift[step];
                    float G = ns_next(&ns);
                    hw_step(&r1, &I1, fmaf(G, sig_st, d), exp_adt, dt);
                    hw_step(&r2, &I2, fmaf(-G, sig_st, d), exp_adt, dt);
                }
                float P1 = bc[i].A * mufu_ex2((r1 * bc[i].negB) * LOG2E_F);
                float P2 = bc[i].A * mufu_ex2((r2 * bc[i].negB) * LOG2E_F);
                float d1 = mufu_ex2(I1 * -LOG2E_F);
                float d2 = mufu_ex2(I2 * -LOG2E_F);
                float x1 = d1 * fmaxf(0.0f, (P1 - caps[i].K) * sgn);
                float x2 = d2 * fmaxf(0.0f, (P2 - caps[i].K) * sgn);
                double X = (double)(caps[i].N * (x1 + x2));
                double Y = (double)(caps[i].N * (P1 * d1 + P2 * d2));
                double* m = loc + 5 * i;
                m[0] += X; m[1] += Y; m[2] += X * X; m[3] += Y * Y; m[4] += X * Y;
                Xs += X;
                Ys += Y;
            }
            double* m = loc + 5 * n;
            m[0] += Xs; m[1] += Ys; m[2] += Xs * Xs; m[3] += Ys * Ys; m[4] += Xs * Ys;
        }
#pragma omp critical
        {
            for (int k = 0; k < nq; k++) mom[k] += loc[k];
        }
        free(loc);
    }
    free(bc);
    FTZ_SCOPE_END
}
