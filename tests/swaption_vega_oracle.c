/*
 * tests/swaption_vega_oracle.c -- TEST INFRASTRUCTURE (CPU oracle of the book vega), not product code.
 *
 * The estimator of hw1f_swaptions_vega restated on the CPU: the book of swaption_oracle.c priced in three sigma
 * scenarios -- sigma, sigma - eps, sigma + eps -- stepped on the SAME normals in reference order (hw_step, libm in place
 * of MUFU).  Each scenario has its own drift (the base table of sigma; the shifted tables of sigma -/+ eps built with
 * fd_theta_a1 := theta_a1, so that every bumped model keeps the curve), its own sig_st and its own bond plans
 * bond_setup(sigma_s, ...).  It is a separate translation unit that includes the oracle's own source, like
 * swaption_oracle.c.  Built by tests/swaption_vega_oracle.py with the flags of oracle/Makefile.
 *
 * mom[11 (n + 1)]: [0, 5 (n + 1)) the moments of orc_swaption_moments (same float sequence, same accumulation), then per
 * option and then for the book six sums over antithetic PAIRS: X-, X-^2, X+, X+^2, D, D^2 with X_s = N (x_s(+G) +
 * x_s(-G)) in float and D = X+ - X- formed in float per pair.  The book's X_s and D are the sums over the options.
 * aux[2][n + 1][5] (optional): the five moments X, Y, X^2, Y^2, XY of each bumped scenario, as orc_swaption_moments
 * lays them out, for the comparison bounds.
 */
#include <omp.h>

#include "hw1f_oracle.c"

typedef struct {
    float T_exercise, K, N;
    int32_t kind, step, first_flow, n_flows, reserved;
} orc_swaption;

typedef struct {
    float T, c;
} orc_cash_flow;

void orc_vega_set_threads(int n) { omp_set_num_threads(n); }

/* x = D max(0, s (Bnd - K)) and y = D Bnd of both twins: the float sequence of orc_swaption_moments */
static void book_payoff(const bond_consts* bc, const orc_cash_flow* fl, int nf, float K, float sgn, float r1, float r2,
                        float I1, float I2, float* x1, float* x2, float* y1, float* y2)
{
    float B1 = 0.0f, B2 = 0.0f;
    for (int j = 0; j < nf; j++) {
        const float c = fl[j].c;
        float P1 = bc[j].A * mufu_ex2((r1 * bc[j].negB) * LOG2E_F);
        float P2 = bc[j].A * mufu_ex2((r2 * bc[j].negB) * LOG2E_F);
        B1 = fmaf(c, P1, B1);
        B2 = fmaf(c, P2, B2);
    }
    float d1 = mufu_ex2(I1 * -LOG2E_F);
    float d2 = mufu_ex2(I2 * -LOG2E_F);
    *x1 = d1 * fmaxf(0.0f, (B1 - K) * sgn);
    *x2 = d2 * fmaxf(0.0f, (B2 - K) * sgn);
    *y1 = B1 * d1;
    *y2 = B2 * d2;
}

void orc_swaption_vega_moments(const orc_params* p, float eps, uint64_t seed, uint64_t first_path, int64_t n_pairs,
                               uint64_t offset_normals, const orc_swaption* sw, int n, const orc_cash_flow* flows,
                               const float* P_mkt, const float* f_mkt, double* mom, double* aux)
{
    xw_build_tables();
    FTZ_SCOPE_BEGIN
    const float exp_adt = orc_exp_adt(p), dt = orc_dt(p), r0 = p->r0;
    const int nb = 5 * (n + 1), nq = 11 * (n + 1), na = 10 * (n + 1), n_last = sw[n - 1].step;
    const int ns = p->n_steps;
    /* scenario 0: sigma; 1: sigma - eps; 2: sigma + eps */
    float sig[3], sst[3];
    sig[0] = p->sigma;
    sig[1] = p->sigma - eps;
    sig[2] = p->sigma + eps;
    float* drift = (float*)malloc(3 * (size_t)ns * sizeof(float));
    float* sdrift = (float*)malloc((size_t)ns * sizeof(float));
    orc_drift_tables(p, sig[0], drift, sdrift);
    orc_params q = *p;
    q.fd_theta_a1 = q.theta_a1;
    for (int s = 1; s < 3; s++) orc_shifted_drift_table(&q, sig[s], sig[0], drift + (size_t)s * ns);
    for (int s = 0; s < 3; s++) sst[s] = orc_sig_st(p, sig[s]);
    int n_rows = 0;
    for (int i = 0; i < n; i++) n_rows += sw[i].n_flows;
    bond_consts* bc = (bond_consts*)malloc(3 * (size_t)n_rows * sizeof(bond_consts));
    orc_cash_flow* fl = (orc_cash_flow*)malloc((size_t)n_rows * sizeof(orc_cash_flow));
    int* row0 = (int*)malloc((size_t)n * sizeof(int));
    for (int i = 0, row = 0; i < n; i++) {
        row0[i] = row;
        for (int j = 0; j < sw[i].n_flows; j++, row++) {
            fl[row] = flows[sw[i].first_flow + j];
            for (int s = 0; s < 3; s++)
                bc[(size_t)s * n_rows + row] = bond_setup(p, sig[s], sw[i].T_exercise, fl[row].T, P_mkt, f_mkt);
        }
    }
    for (int k = 0; k < nq; k++) mom[k] = 0.0;
    if (aux)
        for (int k = 0; k < na; k++) aux[k] = 0.0;
#pragma omp parallel
    {
        FTZ_THREAD
        double* loc = (double*)calloc((size_t)(nq + na), sizeof(double));
        double* la = loc + nq;
#pragma omp for schedule(static)
        for (int64_t pq = 0; pq < n_pairs; pq++) {
            normal_stream nst;
            ns_init(&nst, seed, first_path + (uint64_t)pq, offset_normals);
            float r1[3], r2[3], I1[3], I2[3];
            for (int s = 0; s < 3; s++) { r1[s] = r0; r2[s] = r0; I1[s] = 0.0f; I2[s] = 0.0f; }
            double Xs = 0.0, Ys = 0.0, Xms = 0.0, Xps = 0.0, Ds = 0.0, Xa[2] = {0.0, 0.0}, Ya[2] = {0.0, 0.0};
            int step = 0;
            for (int i = 0; i < n; i++) {
                for (; step < sw[i].step && step < n_last; step++) {
                    const float G = ns_next(&nst);
                    for (int s = 0; s < 3; s++) {
                        const float d = drift[(size_t)s * ns + step];
                        hw_step(&r1[s], &I1[s], fmaf(G, sst[s], d), exp_adt, dt);
                        hw_step(&r2[s], &I2[s], fmaf(-G, sst[s], d), exp_adt, dt);
                    }
                }
                const float sgn = sw[i].kind == 0 ? -1.0f : 1.0f, N = sw[i].N;
                float Xf[3];
                for (int s = 0; s < 3; s++) {
                    float x1, x2, y1, y2;
                    book_payoff(bc + (size_t)s * n_rows + row0[i], fl + row0[i], sw[i].n_flows, sw[i].K, sgn, r1[s],
                                r2[s], I1[s], I2[s], &x1, &x2, &y1, &y2);
                    const double X = (double)(N * (x1 + x2));
                    const double Y = (double)(N * (y1 + y2));
                    Xf[s] = N * (x1 + x2);
                    double* m = s == 0 ? loc + 5 * i : la + (size_t)(s - 1) * nb + 5 * i;
                    m[0] += X; m[1] += Y; m[2] += X * X; m[3] += Y * Y; m[4] += X * Y;
                    if (s == 0) {
                        Xs += X;
                        Ys += Y;
                    } else {
                        Xa[s - 1] += X;
                        Ya[s - 1] += Y;
                    }
                }
                const float Df = Xf[2] - Xf[1];
                const double Xm = (double)Xf[1], Xp = (double)Xf[2], D = (double)Df;
                double* v = loc + nb + 6 * i;
                v[0] += Xm; v[1] += Xm * Xm; v[2] += Xp; v[3] += Xp * Xp; v[4] += D; v[5] += D * D;
                Xms += Xm;
                Xps += Xp;
                Ds += D;
            }
            double* m = loc + 5 * n;
            m[0] += Xs; m[1] += Ys; m[2] += Xs * Xs; m[3] += Ys * Ys; m[4] += Xs * Ys;
            double* v = loc + nb + 6 * n;
            v[0] += Xms; v[1] += Xms * Xms; v[2] += Xps; v[3] += Xps * Xps; v[4] += Ds; v[5] += Ds * Ds;
            for (int s = 0; s < 2; s++) {
                double* a = la + (size_t)s * nb + 5 * n;
                a[0] += Xa[s]; a[1] += Ya[s]; a[2] += Xa[s] * Xa[s]; a[3] += Ya[s] * Ya[s]; a[4] += Xa[s] * Ya[s];
            }
        }
#pragma omp critical
        {
            for (int k = 0; k < nq; k++) mom[k] += loc[k];
            if (aux)
                for (int k = 0; k < na; k++) aux[k] += la[k];
        }
        free(loc);
    }
    free(row0);
    free(fl);
    free(bc);
    free(sdrift);
    free(drift);
    FTZ_SCOPE_END
}
