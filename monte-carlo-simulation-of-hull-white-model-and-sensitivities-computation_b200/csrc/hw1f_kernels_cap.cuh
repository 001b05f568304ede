// hw1f_kernels_cap.cuh -- caps and floors: a strip of caplets (zero-coupon bond puts) or floorlets (bond calls) priced
// in ONE simulation pass.  Every path is stepped once to the last reset step and evaluated at every reset step on the way.
//
//   * Segments.  The time loop walks from one reset step to the next.  A segment may start or end in the middle of a
//     Box-Muller pair: the cos half of a pair that a segment opened is kept and consumed first by the next one (the
//     launch's own `lead` -- an odd normal offset -- is such a cached half too).  Every thread of a launch has the same
//     reset steps, so every branch of the walk is warp-uniform.
//   * Arithmetic.  DECOMP = 0 steps r and I of both antithetic twins with the reference's float sequence (hw_step2, drift
//     staged in shared memory, as zbc_kernel).  DECOMP = 1 carries the one noise recursion (h, W) per stream of
//     fast_kernel (groups of five pairs with their decay residual rho5, single pairs with rho1, so that h is exact at
//     every segment end) and rebuilds at reset step k:  r(+/-) = m_k +/- sg h,  I(+/-) = Im_k +/- c q  (m_k, Im_k: the
//     noise-free tables of the engine, uploaded with the caplet table).
//   * Payoff per twin: D = exp(-I), P = A exp(-B r), x = D max(0, s (P - K)) with s = -1 for a caplet (put) and +1 for a
//     floorlet (call) -- multiplying by +-1 is exact, so a floorlet performs the float operations of zbc_payoffs -- and
//     the control y = D P.  Per antithetic PAIR: X = N (x1 + x2), Y = N (y1 + y2).
//   * Moments.  Per caplet and for the strip (X_s = sum_i X_i, Y_s = sum_i Y_i, accumulated in registers along the path):
//     sum X, sum Y, sum X^2, sum Y^2, sum XY over the pairs.  The control varies by 1e-5 of its value at short resets,
//     so the per-reset float warp trees sum Y - c (c = the noise-free Y, computed in the prologue; Y - c is exact since
//     c / 2 <= Y <= 2 c) and the block undoes the centring in double per chunk: the partial rows hold raw moments.
//   * Reduction: float warp trees -> per-warp rows in shared memory -> double block accumulators -> one partial row of
//     5 (n + 1) doubles per block -> tail_kernel (ncur = 0).  Fixed order, no atomics: bit-reproducible.
#pragma once
#include "hw1f_kernels_extra.cuh"

namespace hw1f {

constexpr int kMaxCaplets = 100;   // HW1F_MAX_CAPLETS: 5 (100 + 1) = 505 moments fit the peer mailboxes (kCommMaxCount)

// one caplet as the host uploads it (the bond plan is computed in the kernel's prologue)
struct CapletDev {
    float T_reset, T_pay, K, N;
    float m, Im;        // noise-free short rate and integral at the reset step (engine tables, double -> float)
    int step;           // reset step, non-decreasing over the strip, in [1, n_steps]
    int pad;
};

// per-caplet constants in shared memory
struct CapletSh {
    float A, negB, K, N, m, Im, cen;
    int step;
};

// x = D max(0, sgn (P - K)), y = D P for both twins of both lanes; sgn = +1 is zbc_payoffs' float sequence
__device__ __forceinline__ void caplet_payoffs(const PairState& st, float A, float negB, float K, float sgn, float2& x1,
                                               float2& x2, float2& c1, float2& c2)
{
    const float2 z1 = mul2(mul2(st.r1, splat(negB)), splat(kLog2e));
    const float2 z2 = mul2(mul2(st.r2, splat(negB)), splat(kLog2e));
    const float2 P1 = mul2(splat(A), make_float2(mufu_ex2(z1.x), mufu_ex2(z1.y)));
    const float2 P2 = mul2(splat(A), make_float2(mufu_ex2(z2.x), mufu_ex2(z2.y)));
    const float2 q1 = mul2(st.I1, splat(-kLog2e)), q2 = mul2(st.I2, splat(-kLog2e));
    const float2 d1 = make_float2(mufu_ex2(q1.x), mufu_ex2(q1.y));
    const float2 d2 = make_float2(mufu_ex2(q2.x), mufu_ex2(q2.y));
    c1 = mul2(P1, d1);
    c2 = mul2(P2, d2);
    const float2 g1 = mul2(add2(P1, splat(-K)), splat(sgn)), g2 = mul2(add2(P2, splat(-K)), splat(sgn));
    x1 = mul2(d1, make_float2(fmaxf(0.0f, g1.x), fmaxf(0.0f, g1.y)));
    x2 = mul2(d2, make_float2(fmaxf(0.0f, g2.x), fmaxf(0.0f, g2.y)));
}

// dynamic shared memory of cap_kernel<DECOMP>
__host__ __device__ inline size_t cap_smem_bytes(int decomp, int n_caplets, int n_last)
{
    const size_t nq = 5 * (size_t)(n_caplets + 1);
    size_t b = (size_t)(decomp ? kWin5Words : kWinWords) * 4;
    b += nq * sizeof(double);                                   // bacc
    b += (size_t)kWarps * nq * sizeof(float);                   // wflt
    b += (size_t)n_caplets * sizeof(CapletSh);                  // caplet constants
    if (!decomp) b += (size_t)n_last * sizeof(float);           // drift of steps [0, n_last)
    return b + 64;
}

// partials[block][5 (n_caplets + 1)] doubles: caplet i at 5 i, the strip at 5 n_caplets; sgn = -1 cap, +1 floor.
// caps[n_caplets] with non-decreasing steps >= 1; P_mkt / f_mkt [n_mat] device curves of the bond plans.
template <int DECOMP>
__global__ void __launch_bounds__(kThreads, HW1F_MIN_BLOCKS)
cap_kernel(StreamGeom g, SeedArgs seeds, ModelDev md, ScenDev sc, const CapletDev* __restrict__ caps, int n_caplets,
           const float* __restrict__ P_mkt, const float* __restrict__ f_mkt, float sgn, int lead,
           double* __restrict__ partials)
{
    extern __shared__ __align__(16) uint32_t smem[];
    // the tail kernel behind this launch may become resident once every block has started (hw1f_tail.cuh)
    asm volatile("griddepcontrol.launch_dependents;");
    const int n = n_caplets, nq = 5 * (n + 1);
    const int n_last = caps[n - 1].step;
    uint32_t* win = smem;
    double* bacc = reinterpret_cast<double*>(smem + (DECOMP ? kWin5Words : kWinWords));   // [nq]
    float* wflt = reinterpret_cast<float*>(bacc + nq);                                     // [kWarps][nq]
    CapletSh* cs = reinterpret_cast<CapletSh*>(wflt + kWarps * nq);                       // [n]
    float* drift = reinterpret_cast<float*>(cs + n);                                      // [n_last] (DECOMP = 0)
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;

    for (int k = tid; k < nq; k += kThreads) bacc[k] = 0.0;
    if (!DECOMP)
        for (int i = tid; i < n_last; i += kThreads) drift[i] = sc.drift2[i].x;
    for (int i = tid; i < n; i += kThreads) {
        // the bond plan of hw1f_zbc_cv (compute_plan on the device curves), and the centring constant: Y of the
        // noise-free pair
        const CapletDev c = caps[i];
        const MktPts none{};
        const BondPlan pl = compute_plan(md, sc.sigma, sc.sig_st, c.T_reset, c.T_pay, P_mkt, f_mkt, none, 0);
        PairState ps;
        ps.r1 = ps.r2 = splat(c.m);
        ps.I1 = ps.I2 = splat(c.Im);
        float2 x1, x2, y1, y2;
        caplet_payoffs(ps, pl.A, pl.negB, c.K, sgn, x1, x2, y1, y2);
        CapletSh s;
        s.A = pl.A; s.negB = pl.negB; s.K = c.K; s.N = c.N; s.m = c.m; s.Im = c.Im;
        s.cen = mul_(c.N, add_(y1.x, y2.x));
        s.step = c.step;
        cs[i] = s;
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
        float2 Xs = splat(0.0f), Ys = splat(0.0f);   // strip: sum of X_i and of the centred Y_i
        for (int i = 0; i < n; ++i) {
            const CapletSh c = cs[i];
            int left = c.step - si;
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
                ps.r1 = add2(splat(c.m), dr);
                ps.r2 = add2(splat(c.m), make_float2(-dr.x, -dr.y));
                ps.I1 = add2(splat(c.Im), dI);
                ps.I2 = add2(splat(c.Im), make_float2(-dI.x, -dI.y));
            } else {
                ps.r1 = r1; ps.r2 = r2; ps.I1 = I1; ps.I2 = I2;
            }
            float2 x1, x2, y1, y2;
            caplet_payoffs(ps, c.A, c.negB, c.K, sgn, x1, x2, y1, y2);
            float2 X = mul2(splat(c.N), add2(x1, x2));
            float2 Y = add2(mul2(splat(c.N), add2(y1, y2)), splat(-c.cen));
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
        // per caplet (and the strip): sum the warp rows in double, undo the centring with this chunk's pair count
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
            if (i < n) c = (double)cs[i].cen;
            else
                for (int j = 0; j < n; ++j) c += (double)cs[j].cen;
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
