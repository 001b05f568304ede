// hw1f_kernels_swaption.cuh -- a book of coupon-bond options priced in ONE simulation pass: European swaptions, and cap
// strips as books of one-flow options.  Every path is stepped once to the last exercise step and every option is
// evaluated at its exercise step on the way.  The walk, the book prologue and the moment rows below are shared with
// book_vega_kernel (hw1f_kernels_book_vega.cuh).
//
//   * Walk (exercise_walk).  Segments run from one distinct exercise step to the next (a shared step is a zero-length
//     segment).  A segment may start or end in the middle of a Box-Muller pair: the cos half of a pair that a segment
//     opened is kept and consumed first by the next one (the launch's own `lead` -- an odd normal offset -- is such a
//     cached half too).  Every thread of a launch has the same exercise steps, so every branch of the walk is
//     warp-uniform.
//   * Arithmetic.  DECOMP = 0 steps r and I of the kernel's twin pairs with the reference's float sequence (hw_step2,
//     drift staged in shared memory, as zbc_kernel): the kernel's step functor.  DECOMP = 1 carries the one noise
//     recursion (h, W) per stream of fast_kernel (groups of five pairs with their decay residual rho5, single pairs with
//     rho1, so that h is exact at every segment end) and rebuilds at exercise step k:  r(+/-) = m_k +/- sg h,
//     I(+/-) = Im_k +/- c q  (m_k, Im_k: the noise-free tables of the engine, uploaded with the option table).
//   * Payoff per twin: D = exp(-I), Bnd = sum_j c_j A_j exp(-B_j r) accumulated in flow order (one fused multiply-add
//     per flow), x = D max(0, s (Bnd - K)) with s = -1 payer (put on the bond) and +1 receiver (call) -- multiplying by
//     +-1 is exact -- and the control y = D Bnd.  Per antithetic PAIR: X = N (x1 + x2), Y = N (y1 + y2).  A caplet is
//     a one-flow option with c = 1: fma(1, P, 0) = P, so it performs the float operations of a single bond option.
//   * Moments.  Per option and for the book (X_s = sum_i X_i, Y_s = sum_i Y_i, accumulated in registers along the
//     path): sum X, sum Y, sum X^2, sum Y^2, sum XY over the pairs.  The control varies by 1e-5 of its value at short
//     exercise dates, so the float warp trees sum Y - c (c = the noise-free Y, computed in the prologue; Y - c is exact
//     since c / 2 <= Y <= 2 c) and the block undoes the centring in double per chunk: the partial rows hold raw moments.
//   * Reduction: float warp trees -> per-warp rows in shared memory -> double block accumulators -> one partial row of
//     5 (n + 1) doubles per block -> tail_kernel (ncur = 0).  Fixed order, no atomics: bit-reproducible.
#pragma once
#include "hw1f_kernels_extra.cuh"
#include "hw1f_kernels_fast.cuh"   // FastState

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

// x = D max(0, sgn (Bnd - K)), y = D Bnd for both twins of both lanes, Bnd = sum_j c_j A_j ex2(negB_j r log2e) over
// the option's flows fl[0, nf).  f0 = fl[0], passed by value so that the walk can load it long before it is used.
__device__ __forceinline__ void swaption_payoffs(const PairState& st, const SwFlowSh& f0, const SwFlowSh* __restrict__ fl,
                                                 int nf, float K, float sgn, float2& x1, float2& x2, float2& c1,
                                                 float2& c2)
{
    float2 B1 = splat(0.0f), B2 = splat(0.0f);
    auto add_flow = [&](const SwFlowSh& f) {
        const float2 z1 = mul2(mul2(st.r1, splat(f.negB)), splat(kLog2e));
        const float2 z2 = mul2(mul2(st.r2, splat(f.negB)), splat(kLog2e));
        const float2 P1 = mul2(splat(f.A), make_float2(mufu_ex2(z1.x), mufu_ex2(z1.y)));
        const float2 P2 = mul2(splat(f.A), make_float2(mufu_ex2(z2.x), mufu_ex2(z2.y)));
        B1 = fma2(splat(f.c), P1, B1);
        B2 = fma2(splat(f.c), P2, B2);
    };
    add_flow(f0);
    for (int j = 1; j < nf; ++j) add_flow(fl[j]);
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

// the book's constants in shared memory: the bond plan of hw1f_zbc_cv for every flow P(T_e, T_j) into fs, then every
// option's constants into ss with its centring constant, Y of the noise-free pair.  per_flow(j, f) runs beside each
// flow's plan, before the barrier between the two.
template <typename PerFlow>
__device__ __forceinline__ void book_prologue(const ModelDev& md, const ScenDev& sc, const SwaptionDev* __restrict__ sw,
                                              int n, const SwFlowDev* __restrict__ flows, int n_rows,
                                              const float* __restrict__ P_mkt, const float* __restrict__ f_mkt,
                                              SwFlowSh* fs, SwaptionSh* ss, PerFlow&& per_flow)
{
    const MktPts none{};
    for (int j = threadIdx.x; j < n_rows; j += kThreads) {
        const SwFlowDev f = flows[j];
        const BondPlan pl = compute_plan(md, sc.sigma, sc.sig_st, f.T_e, f.T, P_mkt, f_mkt, none, 0);
        SwFlowSh s;
        s.A = pl.A; s.negB = pl.negB; s.c = f.c;
        fs[j] = s;
        per_flow(j, f);
    }
    __syncthreads();
    for (int i = threadIdx.x; i < n; i += kThreads) {
        const SwaptionDev o = sw[i];
        PairState ps;
        ps.r1 = ps.r2 = splat(o.m);
        ps.I1 = ps.I2 = splat(o.Im);
        float2 x1, x2, y1, y2;
        swaption_payoffs(ps, fs[o.f0], fs + o.f0, o.nf, o.K, o.sgn, x1, x2, y1, y2);
        SwaptionSh s;
        s.K = o.K; s.N = o.N; s.sgn = o.sgn; s.m = o.m; s.Im = o.Im;
        s.cen = mul_(o.N, add_(y1.x, y2.x));
        s.step = o.step; s.f0 = o.f0; s.nf = o.nf;
        ss[i] = s;
    }
}

// One chunk's walk over the book's exercise steps ss[0, n): at_exercise(i, o, f0, st) evaluates option i = o at its
// step, f0 = fs[o.f0] its first flow row.  Both rows are loaded before the segment is stepped, so that neither load's
// latency (the flow row's address depends on the option row) is exposed at the exercise step.
// Reference order: ref_step(G, si) steps the kernel's twin pairs on the normals G with drift index si.  Decomposed: the
// walk carries the noise state st = (h, W) and never calls ref_step.
template <int DECOMP, typename RefStep, typename AtExercise>
__device__ __forceinline__ void exercise_walk(ThreadStreams& t, const ModelDev& md, const SwaptionSh* ss,
                                              const SwFlowSh* fs, int n, int lead,
                                              RefStep&& ref_step, AtExercise&& at_exercise)
{
    const float2 e2 = splat(md.exp_adt), ee2 = splat(md.exp_2adt);
    FastState st;
    st.h = splat(0.0f);
    st.W = splat(0.0f);
    int si = 0;   // steps taken (reference order: drift index)
    auto step1 = [&](float2 G) {
        if (DECOMP) {
            st.W = add2(st.W, G);
            st.h = fma2(st.h, e2, G);
        } else {
            ref_step(G, si);
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
    for (int i = 0; i < n; ++i) {
        const SwaptionSh o = ss[i];
        const SwFlowSh f0 = fs[o.f0];
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
        at_exercise(i, o, f0, st);
    }
}

// decomposed: both twins of one sigma scenario from the shared noise state, r(+/-) = m +/- sg h, I(+/-) = Im +/- c q
__device__ __forceinline__ PairState rebuild_twins(float2 h, float2 q, float m, float Im, float sg, float c)
{
    const float2 dr = mul2(h, splat(sg)), dI = mul2(q, splat(c));
    PairState ps;
    ps.r1 = add2(splat(m), dr);
    ps.r2 = add2(splat(m), make_float2(-dr.x, -dr.y));
    ps.I1 = add2(splat(Im), dI);
    ps.I2 = add2(splat(Im), make_float2(-dI.x, -dI.y));
    return ps;
}

// sum X, sum Y, sum X^2, sum Y^2, sum XY of the warp through float warp trees into row[0, 5) of the warp's rows
__device__ __forceinline__ void write_moments5(float* row, float2 X, float2 Y, int lane)
{
    const float sX = warp_sum_pair(add_(X.x, X.y), add_(Y.x, Y.y), lane);
    const float sQ = warp_sum_pair(fma_(X.x, X.x, mul_(X.y, X.y)), fma_(Y.x, Y.x, mul_(Y.y, Y.y)), lane);
    const float sXY = warp_sum(fma_(X.x, Y.x, mul_(X.y, Y.y)));
    row += (lane & 16) ? 1 : 0;
    if ((lane & 15) == 0) { row[0] = sX; row[2] = sQ; }
    if (lane == 0) row[4] = sXY;
}

// per option (and the book at row n): sum the five-moment warp rows (stride nq) in double and undo the centring with
// the chunk's pair count into bacc[5 (n + 1)]
__device__ __forceinline__ void fold_moments5(const StreamGeom& g, unsigned long long chunk, const float* wflt, int nq,
                                              const SwaptionSh* ss, int n, double* bacc)
{
    const unsigned long long base = (g.chunk0 + chunk) << kChunkLog2;
    const unsigned long long lo = base > g.first_path ? base : g.first_path;
    const unsigned long long hi = (base + kChunk < g.first_path + g.n_paths) ? base + kChunk : g.first_path + g.n_paths;
    const double nv = (double)(hi - lo);
    for (int i = threadIdx.x; i <= n; i += kThreads) {
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
    book_prologue(md, sc, sw, n, flows, n_rows, P_mkt, f_mkt, fs, ss, [](int, const SwFlowDev&) {});

    const float2 e2 = splat(md.exp_adt), hdt2 = splat(mul_(0.5f, md.dt));
    const float2 sgP = splat(sc.sig_st), sgM = splat(-sc.sig_st);
    const float cI = mul_(mul_(0.5f, md.dt), sc.sig_st);   // FastScen::c

    asm volatile("griddepcontrol.wait;" ::: "memory");   // the per-launch table U of prep_lo_kernel

    for (unsigned long long chunk = blockIdx.x; chunk < g.n_chunks; chunk += gridDim.x) {
        ThreadStreams t = derive_streams<DECOMP ? 5 : 4>(g, seeds, 0, chunk, win);   // contains the __syncthreads()
        const float2 mask = make_float2(t.validA ? 1.0f : 0.0f, t.validB ? 1.0f : 0.0f);
        const bool full = __syncthreads_and(t.validA && t.validB);

        PairState tw;   // reference order: r, I of both twins
        tw.r1 = tw.r2 = splat(md.r0);
        tw.I1 = tw.I2 = splat(0.0f);
        auto ref_step = [&](float2 G, int si) {
            const float2 d = splat(drift[si]);
            hw_step2(tw.r1, tw.I1, fma2(G, sgP, d), e2, hdt2);
            hw_step2(tw.r2, tw.I2, fma2(G, sgM, d), e2, hdt2);
        };
        float2 Xs = splat(0.0f), Ys = splat(0.0f);   // book: sum of X_i and of the centred Y_i
        exercise_walk<DECOMP>(t, md, ss, fs, n, lead, ref_step,
                              [&](int i, const SwaptionSh& o, const SwFlowSh& f0, const FastState& st) {
            const PairState ps = DECOMP ? rebuild_twins(st.h, st.q(md.qA, md.qB), o.m, o.Im, sc.sig_st, cI) : tw;
            float2 x1, x2, y1, y2;
            swaption_payoffs(ps, f0, fs + o.f0, o.nf, o.K, o.sgn, x1, x2, y1, y2);
            float2 X = mul2(splat(o.N), add2(x1, x2));
            float2 Y = add2(mul2(splat(o.N), add2(y1, y2)), splat(-o.cen));
            if (!full) { X = mul2(X, mask); Y = mul2(Y, mask); }   // block-uniform: ragged edge chunks only
            Xs = add2(Xs, X);
            Ys = add2(Ys, Y);
            write_moments5(wflt + warp * nq + 5 * i, X, Y, lane);
        });
        write_moments5(wflt + warp * nq + 5 * n, Xs, Ys, lane);
        __syncthreads();
        fold_moments5(g, chunk, wflt, nq, ss, n, bacc);
    }
    __syncthreads();
    double* out = partials + (size_t)blockIdx.x * nq;
    for (int k = tid; k < nq; k += kThreads) out[k] = bacc[k];
}

}  // namespace hw1f
