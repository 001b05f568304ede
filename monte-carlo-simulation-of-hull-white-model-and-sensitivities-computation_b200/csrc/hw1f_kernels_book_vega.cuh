// hw1f_kernels_book_vega.cuh -- vega of a book of coupon-bond options (European swaptions, cap strips): the book priced
// in three sigma scenarios -- sigma, sigma - eps, sigma + eps -- on ONE set of normals, in ONE simulation pass.  The
// estimator is the common-random-number central difference of run_finite_difference (src/3:400-446); every bumped
// model keeps the initial curve through its own shifted drift table.
//
//   * Walk: exercise_walk of swaption_kernel (hw1f_kernels_swaption.cuh), with its book prologue and moment rows.  Its
//     step functor here steps three twin pairs with hw_step2 in reference order (DECOMP = 0), one per scenario, each on
//     its own drift table (all three staged in shared memory).  DECOMP = 1 carries the one noise recursion (h, W) all
//     scenarios share and rebuilds, at an exercise step k, r_s(+/-) = m_s,k +/- sg_s h and I_s(+/-) = Im_s,k +/- c_s q
//     with q computed once: a bumped scenario costs its payoffs, not another pass over the paths.
//   * Base scenario: the float operations of swaption_kernel -- swaption_payoffs, the same warp trees, the same Y
//     centring and the same per-chunk double accumulation into its own partial row of 5 (n + 1) doubles -- so that its
//     moments equal hw1f_swaptions bit for bit.
//   * Bumped scenarios: the payoff x of swaption_payoffs with the bond plans A_s of sigma_s (negB and c do not depend on
//     sigma).  Per antithetic pair X_s = N (x_s(+G) + x_s(-G)) and D = X_+ - X_-, formed in float per pair before any
//     sum: D is about 2 eps vega, ~1e-3 of X, and a difference of two sums would lose it.  Per option and for the book
//     (X_s summed over the options, D_book = sum_i D_i): sum X_-, X_-^2, X_+, X_+^2, D, D^2 (not centred) through float
//     warp trees into a second partial row of 6 (n + 1) doubles per block.
//   * Reduction: each of the two partial rows goes through tail_kernel (ncur = 0) on its own, so that the base rows are
//     reduced exactly as hw1f_swaptions reduces them (the tail splits the rows by the vector length).  Fixed order, no
//     atomics: bit-reproducible.
#pragma once
#include "hw1f_kernels_swaption.cuh"

namespace hw1f {

// the two bumped scenarios: [0] sigma - eps, [1] sigma + eps
struct BookVegaScen {
    float sigma[2], sig_st[2];
    const float* drift[2];   // [n_steps] shifted drift tables (reference order only)
};

// per-option noise-free short rate and integral of the bumped scenarios at the exercise step
struct BookVegaOptDev {
    float m[2], Im[2];
};

// x = D max(0, sgn (Bnd - K)) for both twins of both lanes of the two bumped scenarios: swaption_payoffs' float
// sequence for x, with the bond plans A_s = fa[j].x (sigma - eps) / fa[j].y (sigma + eps)
__device__ __forceinline__ void bumped_payoffs(const PairState& sm, const PairState& sp, const SwFlowSh* __restrict__ fl,
                                               const float2* __restrict__ fa, int nf, float K, float sgn, float2& xm1,
                                               float2& xm2, float2& xp1, float2& xp2)
{
    float2 Bm1 = splat(0.0f), Bm2 = splat(0.0f), Bp1 = splat(0.0f), Bp2 = splat(0.0f);
    for (int j = 0; j < nf; ++j) {
        const SwFlowSh f = fl[j];
        const float2 A = fa[j];
        const float2 zm1 = mul2(mul2(sm.r1, splat(f.negB)), splat(kLog2e));
        const float2 zm2 = mul2(mul2(sm.r2, splat(f.negB)), splat(kLog2e));
        const float2 zp1 = mul2(mul2(sp.r1, splat(f.negB)), splat(kLog2e));
        const float2 zp2 = mul2(mul2(sp.r2, splat(f.negB)), splat(kLog2e));
        Bm1 = fma2(splat(f.c), mul2(splat(A.x), make_float2(mufu_ex2(zm1.x), mufu_ex2(zm1.y))), Bm1);
        Bm2 = fma2(splat(f.c), mul2(splat(A.x), make_float2(mufu_ex2(zm2.x), mufu_ex2(zm2.y))), Bm2);
        Bp1 = fma2(splat(f.c), mul2(splat(A.y), make_float2(mufu_ex2(zp1.x), mufu_ex2(zp1.y))), Bp1);
        Bp2 = fma2(splat(f.c), mul2(splat(A.y), make_float2(mufu_ex2(zp2.x), mufu_ex2(zp2.y))), Bp2);
    }
    auto x_of = [&](float2 B, float2 I) {
        const float2 q = mul2(I, splat(-kLog2e));
        const float2 d = make_float2(mufu_ex2(q.x), mufu_ex2(q.y));
        const float2 g = mul2(add2(B, splat(-K)), splat(sgn));
        return mul2(d, make_float2(fmaxf(0.0f, g.x), fmaxf(0.0f, g.y)));
    };
    xm1 = x_of(Bm1, sm.I1);
    xm2 = x_of(Bm2, sm.I2);
    xp1 = x_of(Bp1, sp.I1);
    xp2 = x_of(Bp2, sp.I2);
}

// dynamic shared memory of book_vega_kernel<DECOMP>; n_rows = sum of the options' n_flows
__host__ __device__ inline size_t book_vega_smem_bytes(int decomp, int n_swaptions, int n_rows, int n_last)
{
    const size_t nq = 11 * (size_t)(n_swaptions + 1);
    size_t b = (size_t)(decomp ? kWin5Words : kWinWords) * 4;
    b += nq * sizeof(double);                                   // bacc
    b += (size_t)kWarps * nq * sizeof(float);                   // wflt
    b += (size_t)n_rows * sizeof(float2);                       // bumped bond plans A
    b += (size_t)n_swaptions * sizeof(BookVegaOptDev);          // bumped noise-free tables at the exercise steps
    b += (size_t)n_swaptions * sizeof(SwaptionSh);              // option constants
    b += (size_t)n_rows * sizeof(SwFlowSh);                     // flow plans
    if (!decomp) b += 3 * (size_t)n_last * sizeof(float);       // drift of steps [0, n_last), three scenarios
    return b + 64;
}

// sum X-, X-^2, X+, X+^2, D, D^2 of the warp through float warp trees into row[0, 6) of the warp's rows
__device__ __forceinline__ void write_vega6(float* row, float2 Xm, float2 Xp, float2 D, int lane)
{
    const float sm = warp_sum_pair(add_(Xm.x, Xm.y), fma_(Xm.x, Xm.x, mul_(Xm.y, Xm.y)), lane);
    const float sp = warp_sum_pair(add_(Xp.x, Xp.y), fma_(Xp.x, Xp.x, mul_(Xp.y, Xp.y)), lane);
    const float sd = warp_sum_pair(add_(D.x, D.y), fma_(D.x, D.x, mul_(D.y, D.y)), lane);
    row += (lane & 16) ? 1 : 0;
    if ((lane & 15) == 0) { row[0] = sm; row[2] = sp; row[4] = sd; }
}

// partials[block][5 (n + 1)]: the base moments in the layout of swaption_kernel; partials_v[block][6 (n + 1)]: option i
// at 6 i, the book at 6 n.  sw, flows, P_mkt, f_mkt as swaption_kernel; bo[n] the bumped noise-free tables.
// One block per SM: 128 registers for the three scenarios' state and payoffs.
template <int DECOMP>
__global__ void __launch_bounds__(kThreads, 1)
book_vega_kernel(StreamGeom g, SeedArgs seeds, ModelDev md, ScenDev sc, BookVegaScen bv, const SwaptionDev* __restrict__ sw,
                 const BookVegaOptDev* __restrict__ bo, int n, const SwFlowDev* __restrict__ flows, int n_rows,
                 const float* __restrict__ P_mkt, const float* __restrict__ f_mkt, int lead,
                 double* __restrict__ partials, double* __restrict__ partials_v)
{
    extern __shared__ __align__(16) uint32_t smem[];
    // the tail kernel behind this launch may become resident once every block has started (hw1f_tail.cuh)
    asm volatile("griddepcontrol.launch_dependents;");
    const int nb = 5 * (n + 1), nv = 6 * (n + 1), nq = nb + nv;
    const int n_last = sw[n - 1].step;
    uint32_t* win = smem;
    double* bacc = reinterpret_cast<double*>(smem + (DECOMP ? kWin5Words : kWinWords));   // [nq]: base, then vega
    float* wflt = reinterpret_cast<float*>(bacc + nq);                                     // [kWarps][nq]
    float2* fa = reinterpret_cast<float2*>(wflt + kWarps * nq);                            // [n_rows] (A-, A+)
    BookVegaOptDev* bs = reinterpret_cast<BookVegaOptDev*>(fa + n_rows);                  // [n]
    SwaptionSh* ss = reinterpret_cast<SwaptionSh*>(bs + n);                               // [n]
    SwFlowSh* fs = reinterpret_cast<SwFlowSh*>(ss + n);                                   // [n_rows]
    float* drift = reinterpret_cast<float*>(fs + n_rows);                                 // [3][n_last] (DECOMP = 0)
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;

    for (int k = tid; k < nq; k += kThreads) bacc[k] = 0.0;
    if (!DECOMP)
        for (int i = tid; i < n_last; i += kThreads) {
            drift[i] = sc.drift2[i].x;
            drift[n_last + i] = bv.drift[0][i];
            drift[2 * n_last + i] = bv.drift[1][i];
        }
    for (int i = tid; i < n; i += kThreads) bs[i] = bo[i];   // bs and fa: published by book_prologue's barrier
    const MktPts none{};
    book_prologue(md, sc, sw, n, flows, n_rows, P_mkt, f_mkt, fs, ss, [&](int j, const SwFlowDev& f) {
        // the bumped bond plans of P(T_e, T_j): B (so negB) does not depend on sigma
        const BondPlan pm = compute_plan(md, bv.sigma[0], bv.sig_st[0], f.T_e, f.T, P_mkt, f_mkt, none, 0);
        const BondPlan pp = compute_plan(md, bv.sigma[1], bv.sig_st[1], f.T_e, f.T, P_mkt, f_mkt, none, 0);
        fa[j] = make_float2(pm.A, pp.A);
    });

    const float2 e2 = splat(md.exp_adt), hdt2 = splat(mul_(0.5f, md.dt));
    const float sg[3] = {sc.sig_st, bv.sig_st[0], bv.sig_st[1]};   // sigma, sigma - eps, sigma + eps
    float cI[3];                                                    // FastScen::c of each
#pragma unroll
    for (int s = 0; s < 3; ++s) cI[s] = mul_(mul_(0.5f, md.dt), sg[s]);

    asm volatile("griddepcontrol.wait;" ::: "memory");   // the per-launch table U of prep_lo_kernel

    for (unsigned long long chunk = blockIdx.x; chunk < g.n_chunks; chunk += gridDim.x) {
        ThreadStreams t = derive_streams<DECOMP ? 5 : 4>(g, seeds, 0, chunk, win);   // contains the __syncthreads()
        const float2 mask = make_float2(t.validA ? 1.0f : 0.0f, t.validB ? 1.0f : 0.0f);
        const bool full = __syncthreads_and(t.validA && t.validB);

        PairState tw[3];   // reference order: r, I of both twins of the three scenarios
#pragma unroll
        for (int s = 0; s < 3; ++s) {
            tw[s].r1 = tw[s].r2 = splat(md.r0);
            tw[s].I1 = tw[s].I2 = splat(0.0f);
        }
        auto ref_step = [&](float2 G, int si) {
#pragma unroll
            for (int s = 0; s < 3; ++s) {
                const float2 d = splat(drift[s * n_last + si]);
                hw_step2(tw[s].r1, tw[s].I1, fma2(G, splat(sg[s]), d), e2, hdt2);
                hw_step2(tw[s].r2, tw[s].I2, fma2(G, splat(-sg[s]), d), e2, hdt2);
            }
        };
        float2 Xs = splat(0.0f), Ys = splat(0.0f);                       // book: sum of X_i and of the centred Y_i
        float2 Xms = splat(0.0f), Xps = splat(0.0f), Ds = splat(0.0f);   // book: sums of X-_i, X+_i, D_i
        exercise_walk<DECOMP>(t, md, ss, fs, n, lead, ref_step,
                              [&](int i, const SwaptionSh& o, const SwFlowSh& f0, const FastState& st) {
            PairState ps = tw[0], pm = tw[1], pp = tw[2];
            if (DECOMP) {
                const float2 q = st.q(md.qA, md.qB);
                const BookVegaOptDev b = bs[i];
                ps = rebuild_twins(st.h, q, o.m, o.Im, sg[0], cI[0]);
                pm = rebuild_twins(st.h, q, b.m[0], b.Im[0], sg[1], cI[1]);
                pp = rebuild_twins(st.h, q, b.m[1], b.Im[1], sg[2], cI[2]);
            }
            float2 x1, x2, y1, y2;
            swaption_payoffs(ps, f0, fs + o.f0, o.nf, o.K, o.sgn, x1, x2, y1, y2);
            float2 X = mul2(splat(o.N), add2(x1, x2));
            float2 Y = add2(mul2(splat(o.N), add2(y1, y2)), splat(-o.cen));
            float2 xm1, xm2, xp1, xp2;
            bumped_payoffs(pm, pp, fs + o.f0, fa + o.f0, o.nf, o.K, o.sgn, xm1, xm2, xp1, xp2);
            float2 Xm = mul2(splat(o.N), add2(xm1, xm2));
            float2 Xp = mul2(splat(o.N), add2(xp1, xp2));
            if (!full) {   // block-uniform: ragged edge chunks only
                X = mul2(X, mask); Y = mul2(Y, mask);
                Xm = mul2(Xm, mask); Xp = mul2(Xp, mask);
            }
            const float2 D = add2(Xp, make_float2(-Xm.x, -Xm.y));
            Xs = add2(Xs, X);
            Ys = add2(Ys, Y);
            Xms = add2(Xms, Xm);
            Xps = add2(Xps, Xp);
            Ds = add2(Ds, D);
            write_moments5(wflt + warp * nq + 5 * i, X, Y, lane);
            write_vega6(wflt + warp * nq + nb + 6 * i, Xm, Xp, D, lane);
        });
        write_moments5(wflt + warp * nq + 5 * n, Xs, Ys, lane);
        write_vega6(wflt + warp * nq + nb + 6 * n, Xms, Xps, Ds, lane);
        __syncthreads();
        fold_moments5(g, chunk, wflt, nq, ss, n, bacc);
        // bumped scenarios: raw sums, no centring
        for (int k = tid; k < nv; k += kThreads) {
            double acc = (double)wflt[nb + k];
#pragma unroll
            for (int w = 1; w < kWarps; ++w) acc += (double)wflt[w * nq + nb + k];
            bacc[nb + k] += acc;
        }
    }
    __syncthreads();
    double* out = partials + (size_t)blockIdx.x * nb;
    for (int k = tid; k < nb; k += kThreads) out[k] = bacc[k];
    double* out_v = partials_v + (size_t)blockIdx.x * nv;
    for (int k = tid; k < nv; k += kThreads) out_v[k] = bacc[nb + k];
}

}  // namespace hw1f
