// hw1f_kernels_swaption.cuh -- European swaptions: a book of coupon-bond options priced in ONE simulation pass.  Every
// path is stepped once to the last exercise step and every option is evaluated at its exercise step on the way.
//
//   * Walk and arithmetic: those of cap_kernel (hw1f_kernels_cap.cuh), repeated here so that cap_kernel's code stays
//     exactly as it is.  Segments run from one distinct exercise step to the next (a shared step is a zero-length
//     segment); a segment may split a Box-Muller pair, whose cos half the next segment consumes first.  DECOMP = 0 steps
//     r and I of both twins with hw_step2 (drift staged in shared memory); DECOMP = 1 carries the noise recursion (h, W)
//     with the decay residuals rho5 / rho1 and rebuilds r(+/-) = m_k +/- sg h, I(+/-) = Im_k +/- c q at each exercise.
//   * Payoff per twin: D = exp(-I), Bnd = sum_j c_j A_j exp(-B_j r) accumulated in flow order (one fused multiply-add
//     per flow), x = D max(0, s (Bnd - K)) with s = -1 payer (put on the bond) and +1 receiver (call), the control
//     y = D Bnd.  Per antithetic PAIR: X = N (x1 + x2), Y = N (y1 + y2).  A one-flow option with c = 1 performs the
//     float operations of caplet_payoffs (fma(1, P, 0) = P exactly).
//   * Moments: as cap_kernel -- per option and for the book, float warp trees of X and the centred Y (centre: Y of the
//     noise-free pair), per-warp rows, double block accumulators that undo the centring per chunk, one partial row of
//     5 (n + 1) doubles per block, tail_kernel (ncur = 0).  Fixed order, no atomics: bit-reproducible.
#pragma once
#include "hw1f_kernels_cap.cuh"

namespace hw1f {

constexpr int kMaxSwaptions = 100;       // HW1F_MAX_SWAPTIONS: 5 (100 + 1) moments fit the peer mailboxes
constexpr int kMaxSwaptionFlows = 2048;  // HW1F_MAX_SWAPTION_FLOWS

// one option as the host uploads it; its flows are the contiguous rows [f0, f0 + nf) of the uploaded flow table
struct SwaptionDev {
    float T_e, K, N, sgn;   // sgn = -1 payer, +1 receiver
    float m, Im;            // noise-free short rate and integral at the exercise step (engine tables, double -> float)
    int step;               // exercise step, non-decreasing over the book, in [1, n_steps]
    int f0, nf;
    int pad[3];
};

// one flow as the host uploads it: T_e is the exercise date of the option that owns the row
struct SwFlowDev {
    float T_e, T, c, pad;
};

// per-flow bond plan in shared memory: P(T_e, T) = A exp(-B r)
struct SwFlowSh {
    float A, negB, c;
};

// per-option constants in shared memory
struct SwaptionSh {
    float K, N, sgn, m, Im, cen;
    int step, f0, nf;
};

// x = D max(0, sgn (Bnd - K)), y = D Bnd for both twins of both lanes, Bnd = sum_j c_j A_j ex2(negB_j r log2e)
__device__ __forceinline__ void swaption_payoffs(const PairState& st, const SwFlowSh* __restrict__ fl, int nf, float K,
                                                 float sgn, float2& x1, float2& x2, float2& c1, float2& c2)
{
    float2 B1 = splat(0.0f), B2 = splat(0.0f);
    for (int j = 0; j < nf; ++j) {
        const SwFlowSh f = fl[j];
        const float2 z1 = mul2(mul2(st.r1, splat(f.negB)), splat(kLog2e));
        const float2 z2 = mul2(mul2(st.r2, splat(f.negB)), splat(kLog2e));
        const float2 P1 = mul2(splat(f.A), make_float2(mufu_ex2(z1.x), mufu_ex2(z1.y)));
        const float2 P2 = mul2(splat(f.A), make_float2(mufu_ex2(z2.x), mufu_ex2(z2.y)));
        B1 = fma2(splat(f.c), P1, B1);
        B2 = fma2(splat(f.c), P2, B2);
    }
    const float2 q1 = mul2(st.I1, splat(-kLog2e)), q2 = mul2(st.I2, splat(-kLog2e));
    const float2 d1 = make_float2(mufu_ex2(q1.x), mufu_ex2(q1.y));
    const float2 d2 = make_float2(mufu_ex2(q2.x), mufu_ex2(q2.y));
    c1 = mul2(B1, d1);
    c2 = mul2(B2, d2);
    const float2 g1 = mul2(add2(B1, splat(-K)), splat(sgn)), g2 = mul2(add2(B2, splat(-K)), splat(sgn));
    x1 = mul2(d1, make_float2(fmaxf(0.0f, g1.x), fmaxf(0.0f, g1.y)));
    x2 = mul2(d2, make_float2(fmaxf(0.0f, g2.x), fmaxf(0.0f, g2.y)));
}

// dynamic shared memory of swaption_kernel<DECOMP>; n_rows = sum of the options' n_flows
__host__ __device__ inline size_t swaption_smem_bytes(int decomp, int n_swaptions, int n_rows, int n_last)
{
    const size_t nq = 5 * (size_t)(n_swaptions + 1);
    size_t b = (size_t)(decomp ? kWin5Words : kWinWords) * 4;
    b += nq * sizeof(double);                                   // bacc
    b += (size_t)kWarps * nq * sizeof(float);                   // wflt
    b += (size_t)n_swaptions * sizeof(SwaptionSh);              // option constants
    b += (size_t)n_rows * sizeof(SwFlowSh);                     // flow plans
    if (!decomp) b += (size_t)n_last * sizeof(float);           // drift of steps [0, n_last)
    return b + 64;
}

// partials[block][5 (n + 1)] doubles: option i at 5 i, the book at 5 n.  sw[n] with non-decreasing steps >= 1;
// flows[n_rows]; P_mkt / f_mkt [n_mat] device curves of the bond plans.
template <int DECOMP>
__global__ void __launch_bounds__(kThreads, HW1F_MIN_BLOCKS)
swaption_kernel(StreamGeom g, SeedArgs seeds, ModelDev md, ScenDev sc, const SwaptionDev* __restrict__ sw, int n,
                const SwFlowDev* __restrict__ flows, int n_rows, const float* __restrict__ P_mkt,
                const float* __restrict__ f_mkt, int lead, double* __restrict__ partials)
{
    extern __shared__ __align__(16) uint32_t smem[];
    // the tail kernel behind this launch may become resident once every block has started (hw1f_tail.cuh)
    asm volatile("griddepcontrol.launch_dependents;");
    const int nq = 5 * (n + 1);
    const int n_last = sw[n - 1].step;
    uint32_t* win = smem;
    double* bacc = reinterpret_cast<double*>(smem + (DECOMP ? kWin5Words : kWinWords));   // [nq]
    float* wflt = reinterpret_cast<float*>(bacc + nq);                                     // [kWarps][nq]
    SwaptionSh* ss = reinterpret_cast<SwaptionSh*>(wflt + kWarps * nq);                   // [n]
    SwFlowSh* fs = reinterpret_cast<SwFlowSh*>(ss + n);                                   // [n_rows]
    float* drift = reinterpret_cast<float*>(fs + n_rows);                                 // [n_last] (DECOMP = 0)
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;

    for (int k = tid; k < nq; k += kThreads) bacc[k] = 0.0;
    if (!DECOMP)
        for (int i = tid; i < n_last; i += kThreads) drift[i] = sc.drift2[i].x;
    const MktPts none{};
    for (int j = tid; j < n_rows; j += kThreads) {
        // the bond plan of hw1f_zbc_cv / cap_kernel for P(T_e, T_j)
        const SwFlowDev f = flows[j];
        const BondPlan pl = compute_plan(md, sc.sigma, sc.sig_st, f.T_e, f.T, P_mkt, f_mkt, none, 0);
        SwFlowSh s;
        s.A = pl.A; s.negB = pl.negB; s.c = f.c;
        fs[j] = s;
    }
    __syncthreads();
    for (int i = tid; i < n; i += kThreads) {
        // the centring constant: Y of the noise-free pair
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
    const bool writer = (lane & 15) == 0;

    asm volatile("griddepcontrol.wait;" ::: "memory");   // the per-launch table U of prep_lo_kernel

    for (unsigned long long chunk = blockIdx.x; chunk < g.n_chunks; chunk += gridDim.x) {
        ThreadStreams t = derive_streams<DECOMP ? 5 : 4>(g, seeds, 0, chunk, win);   // contains the __syncthreads()
        const float2 mask = make_float2(t.validA ? 1.0f : 0.0f, t.validB ? 1.0f : 0.0f);
        const bool full = __syncthreads_and(t.validA && t.validB);

        // reference order: r, I of both twins; decomposed: the shared noise state
        float2 r1 = splat(md.r0), r2 = splat(md.r0), I1 = splat(0.0f), I2 = splat(0.0f);
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
            PairState ps;
            if (DECOMP) {
                const float2 q = st.q(md.qA, md.qB);
                const float2 dr = mul2(st.h, splat(sc.sig_st)), dI = mul2(q, splat(cI));
                ps.r1 = add2(splat(o.m), dr);
                ps.r2 = add2(splat(o.m), make_float2(-dr.x, -dr.y));
                ps.I1 = add2(splat(o.Im), dI);
                ps.I2 = add2(splat(o.Im), make_float2(-dI.x, -dI.y));
            } else {
                ps.r1 = r1; ps.r2 = r2; ps.I1 = I1; ps.I2 = I2;
            }
            float2 x1, x2, y1, y2;
            swaption_payoffs(ps, fs + o.f0, o.nf, o.K, o.sgn, x1, x2, y1, y2);
            float2 X = mul2(splat(o.N), add2(x1, x2));
            float2 Y = add2(mul2(splat(o.N), add2(y1, y2)), splat(-o.cen));
            if (!full) { X = mul2(X, mask); Y = mul2(Y, mask); }   // block-uniform: ragged edge chunks only
            Xs = add2(Xs, X);
            Ys = add2(Ys, Y);
            const float sX = warp_sum_pair(add_(X.x, X.y), add_(Y.x, Y.y), lane);
            const float sQ = warp_sum_pair(fma_(X.x, X.x, mul_(X.y, X.y)), fma_(Y.x, Y.x, mul_(Y.y, Y.y)), lane);
            const float sXY = warp_sum(fma_(X.x, Y.x, mul_(X.y, Y.y)));
            float* row = wflt + warp * nq + 5 * i + ((lane & 16) ? 1 : 0);
            if (writer) { row[0] = sX; row[2] = sQ; }
            if (lane == 0) row[4] = sXY;
        }
        {
            const float sX = warp_sum_pair(add_(Xs.x, Xs.y), add_(Ys.x, Ys.y), lane);
            const float sQ = warp_sum_pair(fma_(Xs.x, Xs.x, mul_(Xs.y, Xs.y)), fma_(Ys.x, Ys.x, mul_(Ys.y, Ys.y)), lane);
            const float sXY = warp_sum(fma_(Xs.x, Ys.x, mul_(Xs.y, Ys.y)));
            float* row = wflt + warp * nq + 5 * n + ((lane & 16) ? 1 : 0);
            if (writer) { row[0] = sX; row[2] = sQ; }
            if (lane == 0) row[4] = sXY;
        }
        __syncthreads();
        // per option (and the book): sum the warp rows in double, undo the centring with this chunk's pair count
        const unsigned long long base = (g.chunk0 + chunk) << kChunkLog2;
        const unsigned long long lo = base > g.first_path ? base : g.first_path;
        const unsigned long long hi = (base + kChunk < g.first_path + g.n_paths) ? base + kChunk : g.first_path + g.n_paths;
        const double nv = (double)(hi - lo);
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
            b[1] += s[1] + nv * c;
            b[2] += s[2];
            b[3] += s[3] + 2.0 * c * s[1] + nv * c * c;
            b[4] += s[4] + c * s[0];
        }
    }
    __syncthreads();
    double* out = partials + (size_t)blockIdx.x * nq;
    for (int k = tid; k < nq; k += kThreads) out[k] = bacc[k];
}

}  // namespace hw1f
