// hw1f_kernels_book_vega.cuh -- vega of a book of coupon-bond options (European swaptions, cap strips): the book priced
// in three sigma scenarios -- sigma, sigma - eps, sigma + eps -- on ONE set of normals, in ONE simulation pass.  The
// estimator is the common-random-number central difference of run_finite_difference (src/3:400-446); every bumped
// model keeps the initial curve through its own shifted drift table.
//
//   * Walk: that of swaption_kernel (hw1f_kernels_swaption.cuh), repeated here so that swaption_kernel's code stays
//     exactly as it is.  DECOMP = 0 steps three twin pairs with hw_step2, one per scenario, each on its own drift table
//     (all three staged in shared memory).  DECOMP = 1 carries the one noise recursion (h, W) all scenarios share and
//     rebuilds, at an exercise step k, r_s(+/-) = m_s,k +/- sg_s h and I_s(+/-) = Im_s,k +/- c_s q with q computed once:
//     a bumped scenario costs its payoffs, not another pass over the paths.
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
    const MktPts none{};
    for (int j = tid; j < n_rows; j += kThreads) {
        // the bond plans of P(T_e, T_j) in the three scenarios: B (so negB) does not depend on sigma
        const SwFlowDev f = flows[j];
        const BondPlan pl = compute_plan(md, sc.sigma, sc.sig_st, f.T_e, f.T, P_mkt, f_mkt, none, 0);
        const BondPlan pm = compute_plan(md, bv.sigma[0], bv.sig_st[0], f.T_e, f.T, P_mkt, f_mkt, none, 0);
        const BondPlan pp = compute_plan(md, bv.sigma[1], bv.sig_st[1], f.T_e, f.T, P_mkt, f_mkt, none, 0);
        SwFlowSh s;
        s.A = pl.A; s.negB = pl.negB; s.c = f.c;
        fs[j] = s;
        fa[j] = make_float2(pm.A, pp.A);
    }
    for (int i = tid; i < n; i += kThreads) bs[i] = bo[i];
    __syncthreads();
    for (int i = tid; i < n; i += kThreads) {
        // the centring constant of the base control: Y of the noise-free pair
        const SwaptionDev o = sw[i];
        PairState ps;
        ps.r1 = ps.r2 = splat(o.m);
        ps.I1 = ps.I2 = splat(o.Im);
        float2 x1, x2, y1, y2;
        swaption_payoffs(ps, fs + o.f0, o.nf, o.K, o.sgn, x1, x2, y1, y2);
        SwaptionSh s;
        s.K = o.K; s.N = o.N; s.sgn = o.sgn; s.m = o.m; s.Im = o.Im;
        s.cen = mul_(o.N, add_(y1.x, y2.x));
        s.step = o.step; s.f0 = o.f0; s.nf = o.nf;
        ss[i] = s;
    }

    const float2 e2 = splat(md.exp_adt), ee2 = splat(md.exp_2adt), hdt2 = splat(mul_(0.5f, md.dt));
    const float2 sgP = splat(sc.sig_st), sgM = splat(-sc.sig_st);
    const float cI = mul_(mul_(0.5f, md.dt), sc.sig_st);   // FastScen::c
    float cIb[2];
    float2 sgPb[2], sgMb[2];
#pragma unroll
    for (int s = 0; s < 2; ++s) {
        cIb[s] = mul_(mul_(0.5f, md.dt), bv.sig_st[s]);
        sgPb[s] = splat(bv.sig_st[s]);
        sgMb[s] = splat(-bv.sig_st[s]);
    }
    const bool writer = (lane & 15) == 0;

    asm volatile("griddepcontrol.wait;" ::: "memory");   // the per-launch table U of prep_lo_kernel

    for (unsigned long long chunk = blockIdx.x; chunk < g.n_chunks; chunk += gridDim.x) {
        ThreadStreams t = derive_streams<DECOMP ? 5 : 4>(g, seeds, 0, chunk, win);   // contains the __syncthreads()
        const float2 mask = make_float2(t.validA ? 1.0f : 0.0f, t.validB ? 1.0f : 0.0f);
        const bool full = __syncthreads_and(t.validA && t.validB);

        // reference order: r, I of both twins of the base and of the two bumped scenarios; decomposed: the shared noise
        float2 r1 = splat(md.r0), r2 = splat(md.r0), I1 = splat(0.0f), I2 = splat(0.0f);
        PairState bp[2];
#pragma unroll
        for (int s = 0; s < 2; ++s) {
            bp[s].r1 = bp[s].r2 = splat(md.r0);
            bp[s].I1 = bp[s].I2 = splat(0.0f);
        }
        FastState st;
        st.h = splat(0.0f);
        st.W = splat(0.0f);
        int si = 0;   // steps taken (reference order: drift index)
        auto step1 = [&](float2 G) {
            if (DECOMP) {
                st.W = add2(st.W, G);
                st.h = fma2(st.h, e2, G);
            } else {
                const float2 d = splat(drift[si]);
                hw_step2(r1, I1, fma2(G, sgP, d), e2, hdt2);
                hw_step2(r2, I2, fma2(G, sgM, d), e2, hdt2);
#pragma unroll
                for (int s = 0; s < 2; ++s) {
                    const float2 ds = splat(drift[(s + 1) * n_last + si]);
                    hw_step2(bp[s].r1, bp[s].I1, fma2(G, sgPb[s], ds), e2, hdt2);
                    hw_step2(bp[s].r2, bp[s].I2, fma2(G, sgMb[s], ds), e2, hdt2);
                }
            }
            ++si;
        };
        // reference order: two steps per pair
        auto pairfn = [&](int, float2 ns, float2 nc) { step1(ns); step1(nc); };
        // decomposed: fast_kernel's pair step, the group's decay residual at HW1F_RHO_POS
        auto fpair5 = [&](int j, float2 s, float2 sn, float2 c) {
            const float2 a = fma2(sn, e2, c);
            const float2 b = add2(sn, c);
            if (j == HW1F_RHO_POS) st.h = fma2(st.h, splat(md.rho5), st.h);
            st.h = fma2(s, a, mul2(st.h, ee2));
            st.W = fma2(s, b, st.W);
        };
        auto fpair1 = [&](int, float2 s, float2 sn, float2 c) {
            const float2 a = fma2(sn, e2, c);
            const float2 b = add2(sn, c);
            st.h = fma2(s, a, mul2(st.h, ee2));
            st.W = fma2(s, b, st.W);
        };
        auto advance = [&](int n_pairs) {
            if (DECOMP) {
                int pair = 0, k = 0;
                for (; k + 5 <= n_pairs; k += 5) { run_pairs_parts<5, 0>(t, pair, fpair5); pair += 5; }
                for (; k < n_pairs; ++k) {
                    st.h = fma2(st.h, splat(md.rho1), st.h);
                    run_pairs_parts<1, 0>(t, pair, fpair1);
                    pair += 1;
                }
                si += 2 * n_pairs;
            } else {
                int pair = 0;
                advance_pairs(t, pair, n_pairs, pairfn);
            }
        };

        bool pending = false;          // the cos half of the last pair is still to be stepped
        float2 nc_keep = splat(0.0f);
        if (lead) {                    // the launch starts on the cos half of a pair the previous launch opened
            float2 ns;
            one_pair(t, ns, nc_keep);
            pending = true;
        }
        float2 Xs = splat(0.0f), Ys = splat(0.0f);   // book: sum of X_i and of the centred Y_i
        float2 Xms = splat(0.0f), Xps = splat(0.0f), Ds = splat(0.0f);   // book: sums of X-_i, X+_i, D_i
        for (int i = 0; i < n; ++i) {
            const SwaptionSh o = ss[i];
            int left = o.step - si;
            if (left > 0) {
                if (pending) { step1(nc_keep); pending = false; --left; }
                advance(left >> 1);
                if (left & 1) {
                    float2 ns;
                    one_pair(t, ns, nc_keep);
                    step1(ns);
                    pending = true;
                }
            }
            PairState ps, pb[2];
            if (DECOMP) {
                const float2 q = st.q(md.qA, md.qB);
                const float2 dr = mul2(st.h, splat(sc.sig_st)), dI = mul2(q, splat(cI));
                ps.r1 = add2(splat(o.m), dr);
                ps.r2 = add2(splat(o.m), make_float2(-dr.x, -dr.y));
                ps.I1 = add2(splat(o.Im), dI);
                ps.I2 = add2(splat(o.Im), make_float2(-dI.x, -dI.y));
                const BookVegaOptDev b = bs[i];
#pragma unroll
                for (int s = 0; s < 2; ++s) {
                    const float2 drs = mul2(st.h, splat(bv.sig_st[s])), dIs = mul2(q, splat(cIb[s]));
                    pb[s].r1 = add2(splat(b.m[s]), drs);
                    pb[s].r2 = add2(splat(b.m[s]), make_float2(-drs.x, -drs.y));
                    pb[s].I1 = add2(splat(b.Im[s]), dIs);
                    pb[s].I2 = add2(splat(b.Im[s]), make_float2(-dIs.x, -dIs.y));
                }
            } else {
                ps.r1 = r1; ps.r2 = r2; ps.I1 = I1; ps.I2 = I2;
                pb[0] = bp[0];
                pb[1] = bp[1];
            }
            float2 x1, x2, y1, y2;
            swaption_payoffs(ps, fs + o.f0, o.nf, o.K, o.sgn, x1, x2, y1, y2);
            float2 X = mul2(splat(o.N), add2(x1, x2));
            float2 Y = add2(mul2(splat(o.N), add2(y1, y2)), splat(-o.cen));
            float2 xm1, xm2, xp1, xp2;
            bumped_payoffs(pb[0], pb[1], fs + o.f0, fa + o.f0, o.nf, o.K, o.sgn, xm1, xm2, xp1, xp2);
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
            {
                const float sX = warp_sum_pair(add_(X.x, X.y), add_(Y.x, Y.y), lane);
                const float sQ = warp_sum_pair(fma_(X.x, X.x, mul_(X.y, X.y)), fma_(Y.x, Y.x, mul_(Y.y, Y.y)), lane);
                const float sXY = warp_sum(fma_(X.x, Y.x, mul_(X.y, Y.y)));
                float* row = wflt + warp * nq + 5 * i + ((lane & 16) ? 1 : 0);
                if (writer) { row[0] = sX; row[2] = sQ; }
                if (lane == 0) row[4] = sXY;
            }
            {
                const float sm = warp_sum_pair(add_(Xm.x, Xm.y), fma_(Xm.x, Xm.x, mul_(Xm.y, Xm.y)), lane);
                const float sp = warp_sum_pair(add_(Xp.x, Xp.y), fma_(Xp.x, Xp.x, mul_(Xp.y, Xp.y)), lane);
                const float sd = warp_sum_pair(add_(D.x, D.y), fma_(D.x, D.x, mul_(D.y, D.y)), lane);
                float* row = wflt + warp * nq + nb + 6 * i + ((lane & 16) ? 1 : 0);
                if (writer) { row[0] = sm; row[2] = sp; row[4] = sd; }
            }
        }
        {
            const float sX = warp_sum_pair(add_(Xs.x, Xs.y), add_(Ys.x, Ys.y), lane);
            const float sQ = warp_sum_pair(fma_(Xs.x, Xs.x, mul_(Xs.y, Xs.y)), fma_(Ys.x, Ys.x, mul_(Ys.y, Ys.y)), lane);
            const float sXY = warp_sum(fma_(Xs.x, Ys.x, mul_(Xs.y, Ys.y)));
            float* row = wflt + warp * nq + 5 * n + ((lane & 16) ? 1 : 0);
            if (writer) { row[0] = sX; row[2] = sQ; }
            if (lane == 0) row[4] = sXY;
        }
        {
            const float sm = warp_sum_pair(add_(Xms.x, Xms.y), fma_(Xms.x, Xms.x, mul_(Xms.y, Xms.y)), lane);
            const float sp = warp_sum_pair(add_(Xps.x, Xps.y), fma_(Xps.x, Xps.x, mul_(Xps.y, Xps.y)), lane);
            const float sd = warp_sum_pair(add_(Ds.x, Ds.y), fma_(Ds.x, Ds.x, mul_(Ds.y, Ds.y)), lane);
            float* row = wflt + warp * nq + nb + 6 * n + ((lane & 16) ? 1 : 0);
            if (writer) { row[0] = sm; row[2] = sp; row[4] = sd; }
        }
        __syncthreads();
        // base, per option (and the book): sum the warp rows in double, undo the centring with this chunk's pair count
        const unsigned long long base = (g.chunk0 + chunk) << kChunkLog2;
        const unsigned long long lo = base > g.first_path ? base : g.first_path;
        const unsigned long long hi = (base + kChunk < g.first_path + g.n_paths) ? base + kChunk : g.first_path + g.n_paths;
        const double nvp = (double)(hi - lo);
        for (int i = tid; i <= n; i += kThreads) {
            double s[5];
#pragma unroll
            for (int k = 0; k < 5; ++k) {
                double acc = (double)wflt[5 * i + k];
#pragma unroll
                for (int w = 1; w < kWarps; ++w) acc += (double)wflt[w * nq + 5 * i + k];
                s[k] = acc;
            }
            double c = 0.0;
            if (i < n) c = (double)ss[i].cen;
            else
                for (int j = 0; j < n; ++j) c += (double)ss[j].cen;
            double* b = bacc + 5 * i;
            b[0] += s[0];
            b[1] += s[1] + nvp * c;
            b[2] += s[2];
            b[3] += s[3] + 2.0 * c * s[1] + nvp * c * c;
            b[4] += s[4] + c * s[0];
        }
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
