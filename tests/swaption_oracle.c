/*
 * tests/swaption_oracle.c -- TEST INFRASTRUCTURE (CPU oracle of the swaption book), not product code.
 *
 * The book estimator of hw1f_swaptions restated on the CPU: the reference-order float sequence of orc_zbc_moments
 * (bond_setup per flow, hw_step, libm in place of MUFU) evaluated at every exercise step of each pair of paths.  It is a
 * separate translation unit that includes the oracle's own source, so that it runs the oracle's static RNG, Box-Muller,
 * step and bond-plan code itself instead of a copy of it.  Built by tests/swaption_oracle.py with the flags of
 * oracle/Makefile.
 *
 * One option = a coupon-bond option exercised at T_e, read at step `step` (non-decreasing along the book, >= 1), on the
 * flows flows[first_flow, first_flow + n_flows): Bnd = sum_j c_j A_j exp2(negB_j r log2e) accumulated in flow order
 * with one fused multiply-add per flow, x = D max(0, s (Bnd - K)) with s = -1 payer, +1 receiver, y = D Bnd.
 * mom[5 (n + 1)]: per option and then for the book, sums over antithetic PAIRS of X, Y, X^2, Y^2, XY with
 * X = N (x(+G) + x(-G)), Y = N (y(+G) + y(-G)); the book's X, Y are the sums over the options.
 */
#include "hw1f_oracle.c"

typedef struct {
    float T_exercise, K, N;
    int32_t kind, step, first_flow, n_flows, reserved;
} orc_swaption;

typedef struct {
    float T, c;
} orc_cash_flow;

/* ---- European swaptions ---------------------------------------------------------- */
void orc_swaption_moments(const orc_params* p, float sigma, float sig_st, const float* drift,
                          uint64_t seed, uint64_t first_path, int64_t n_pairs, uint64_t offset_normals,
                          const orc_swaption* sw, int n, const orc_cash_flow* flows, const float* P_mkt,
                          const float* f_mkt, double* mom)
{
    xw_build_tables();
    FTZ_SCOPE_BEGIN
    const float exp_adt = orc_exp_adt(p), dt = orc_dt(p), r0 = p->r0;
    const int nq = 5 * (n + 1), n_last = sw[n - 1].step;
    int n_rows = 0;
    for (int i = 0; i < n; i++) n_rows += sw[i].n_flows;
    /* the bond plan of every (option, flow): P(T_e, T_j) = A exp(-B r) */
    bond_consts* bc = (bond_consts*)malloc((size_t)n_rows * sizeof(bond_consts));
    int* row0 = (int*)malloc((size_t)n * sizeof(int));
    for (int i = 0, row = 0; i < n; i++) {
        row0[i] = row;
        for (int j = 0; j < sw[i].n_flows; j++, row++)
            bc[row] = bond_setup(p, sigma, sw[i].T_exercise, flows[sw[i].first_flow + j].T, P_mkt, f_mkt);
    }
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
                for (; step < sw[i].step && step < n_last; step++) {
                    float d = drift[step];
                    float G = ns_next(&ns);
                    hw_step(&r1, &I1, fmaf(G, sig_st, d), exp_adt, dt);
                    hw_step(&r2, &I2, fmaf(-G, sig_st, d), exp_adt, dt);
                }
                const float sgn = sw[i].kind == 0 ? -1.0f : 1.0f;
                float B1 = 0.0f, B2 = 0.0f;
                for (int j = 0; j < sw[i].n_flows; j++) {
                    const bond_consts* b = &bc[row0[i] + j];
                    const float c = flows[sw[i].first_flow + j].c;
                    float P1 = b->A * mufu_ex2((r1 * b->negB) * LOG2E_F);
                    float P2 = b->A * mufu_ex2((r2 * b->negB) * LOG2E_F);
                    B1 = fmaf(c, P1, B1);
                    B2 = fmaf(c, P2, B2);
                }
                float d1 = mufu_ex2(I1 * -LOG2E_F);
                float d2 = mufu_ex2(I2 * -LOG2E_F);
                float x1 = d1 * fmaxf(0.0f, (B1 - sw[i].K) * sgn);
                float x2 = d2 * fmaxf(0.0f, (B2 - sw[i].K) * sgn);
                double X = (double)(sw[i].N * (x1 + x2));
                double Y = (double)(sw[i].N * (B1 * d1 + B2 * d2));
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
    free(row0);
    free(bc);
    FTZ_SCOPE_END
}
