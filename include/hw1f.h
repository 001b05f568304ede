/*
 * include/hw1f.h -- C ABI of the B200-native Hull-White one-factor Monte Carlo engine.
 *
 * The reference (giulialionetti/Monte-Carlo-simulation-of-Hull-White-model-and-
 * sensitivities-computation) has no FFI: its "operator surface" is the set of
 * kernel launches, __constant__-symbol writes and raw device buffers that its four
 * drivers perform in the same translation unit as main().  Every entry point below
 * names the reference call sites it replaces (paths relative to the reference root).
 *
 * Conventions
 *   - plain C types only; all array arguments are HOST pointers unless the name
 *     starts with d_ (device pointer, used by the *_moments / *_finish pairs that
 *     let a caller put its own collective between simulation and finalisation);
 *   - every function returns an int status (HW1F_OK == 0); nothing calls exit()
 *     (the reference's check_cuda() does, include/common.cuh:114-120);
 *   - "n_paths" is the reference's N_PATHS: the number of RNG subsequences.  The
 *     antithetic kernels simulate 2*n_paths trajectories, like the reference;
 *   - RNG streams are cuRAND-XORWOW compatible: path p of an hw1f_rng created with
 *     (seed, first_path) sees exactly the Gaussians that
 *     curand_init(seed, first_path + p, 0, &st) + curand_normal(&st) would deliver
 *     (include/common.cuh:277-280, :327), starting at the handle's normal offset.
 *     No per-path state array exists; the state is re-derived inside the kernels.
 *   - there is NO CPU fallback: without a CUDA device every compute call fails;
 *   - an engine owns one stream and scratch buffers: it is not thread-safe.  Use one engine
 *     per host thread (engines on the same device share nothing but the GPU).
 */
#ifndef HW1F_H
#define HW1F_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define HW1F_OK 0
#define HW1F_ERR_INVALID 1        /* bad argument                          */
#define HW1F_ERR_CUDA 2           /* a CUDA runtime call failed             */
#define HW1F_ERR_NO_DEVICE 3      /* no usable CUDA device                  */
#define HW1F_ERR_UNSUPPORTED 4    /* configuration outside the engine       */
#define HW1F_ERR_NO_MODEL 5       /* hw1f_set_model() not called yet        */
#define HW1F_ERR_COMM 6           /* moment vector not finite: a peer all-reduce timed out (hw1f_comm_*) */

#define HW1F_ABI_VERSION 1

/* ---- model ------------------------------------------------------------------ */
/* Replaces the compile-time configuration of include/common.cuh:16-39 and the
 * piecewise-linear theta hard-coded at common.cuh:74-76 / :228-230. */
typedef struct hw1f_params {
    float a;            /* H_A      mean reversion                */
    float sigma;        /* H_SIGMA  volatility                    */
    float r0;           /* H_R0     initial short rate            */
    float T_final;      /* T_FINAL                                */
    int32_t n_steps;    /* N_STEPS                                */
    int32_t n_mat;      /* N_MAT    (n_steps % (n_mat-1) == 0)    */
    float theta_a0, theta_b0;   /* theta(t) = a0 + b0 t, t <  theta_break */
    float theta_a1, theta_b1;   /* theta(t) = a1 + b1 t, t >= theta_break */
    float theta_break;
    float fd_theta_a1;  /* constant used by compute_shifted_drift_table for t >= break
                           (0.014 in src/3_sensitivity_analysis.cu:387; quirk kept) */
} hw1f_params;

typedef struct hw1f_engine hw1f_engine; /* one per (process, device): tables, scratch, stream */
typedef struct hw1f_rng hw1f_rng;       /* (seed, first_path, n_paths, normal offset)        */

int hw1f_abi_version(void);
const char* hw1f_status_string(int status);
/* message of the last failure on this engine (never NULL) */
const char* hw1f_last_error(const hw1f_engine* eng);

/* select_gpu() + cudaMalloc of every scratch buffer (common.cuh:122-141; src/1:38-42).
 * device < 0 picks the device with the most free memory like select_gpu(). */
int hw1f_engine_create(int device, hw1f_engine** out);
int hw1f_engine_destroy(hw1f_engine* eng);
/* run on a caller-owned cudaStream_t (NULL = the engine's own stream) */
int hw1f_engine_set_stream(hw1f_engine* eng, void* cuda_stream);
int hw1f_engine_device(const hw1f_engine* eng, int* device);
/* Simulation arithmetic.  Both modes consume bit-identical XORWOW integers and Box-Muller normals.
 *   HW1F_MODE_REFERENCE_ORDER: every path is stepped with the reference's own float sequence
 *       (FFMA, FFMA, FADD, FMUL, FFMA per path-step; include/common.cuh:237-244).
 *   HW1F_MODE_DECOMPOSED (default): the model is linear in the shocks, so the +G/-G twins, the
 *       sigma-bumped twins and the pathwise tangent are all (noise-free part) +/- scale * h with ONE
 *       shared noise recursion h' = h e^{-a dt} + G per stream; per-path values differ from the
 *       reference by float rounding only (~1e-7 relative; north-star tolerance 1e-5). */
#define HW1F_MODE_REFERENCE_ORDER 0
#define HW1F_MODE_DECOMPOSED 1
int hw1f_engine_set_mode(hw1f_engine* eng, int mode);
int hw1f_engine_get_mode(const hw1f_engine* eng, int* mode);
int hw1f_engine_synchronize(hw1f_engine* eng);

/* H_* constants of common.cuh:33-39 */
int hw1f_default_params(hw1f_params* out);
/* compute_constants() + compute_drift_tables(): every cudaMemcpyToSymbol of
 * common.cuh:82-83,98-106 and src/3:416-420,428-432,439-441,453-455,518-520. */
int hw1f_set_model(hw1f_engine* eng, const hw1f_params* p);
/* Configuration space: n_steps must be a multiple of n_mat - 1 (the reference's #error, common.cuh:25-27); any save
 * stride n_steps / (n_mat - 1), even or odd, is supported by the curve entry points (hw1f_bond_curve*,
 * hw1f_vega_fd_recalibrated, hw1f_vega), which need an EVEN normal offset (they start on a Box-Muller pair boundary;
 * HW1F_ERR_UNSUPPORTED with a message otherwise).  Only the fused single-window pass (hw1f_fused*) needs an even
 * stride and n_steps_S1 on the maturity grid.  hw1f_zbc_cv*, hw1f_vega_pathwise*, hw1f_vega_fd and hw1f_sample_paths
 * take any step count and offset parity.
 * Size limits: n_mat in [3, 1024], n_steps in [2, 8192].  Every single-scenario entry point works over that whole range
 * (tests/test_gpu_parity.py::test_other_model_parameters runs 2 x 3, 8184 x 1024 and 1023 x 1024 against the oracle); the
 * two-scenario curve passes (hw1f_vega, hw1f_vega_fd_recalibrated, hw1f_fused*) keep per-warp rows of 2 x 2 x n_mat sums or
 * both drift tables in shared memory and return HW1F_ERR_UNSUPPORTED ("model too large for shared memory") on the largest
 * grids (n_mat beyond about 700 in decomposed mode) -- never a wrong result (tools/extreme_configs.py walks every entry point
 * over the corner configurations in both modes). */
int hw1f_get_model(const hw1f_engine* eng, hw1f_params* out);
/* host copies of the derived constants, for callers that print them */
typedef struct hw1f_constants {
    float dt, mat_spacing, exp_adt, sig_st;
    int32_t save_stride;
} hw1f_constants;
int hw1f_get_constants(const hw1f_engine* eng, hw1f_constants* out);
/* which = 0: drift table at sigma (common.cuh:73-76); 1: sensitivity drift table (common.cuh:79-80);
 * 2: shifted drift table for sigma vs. the model sigma (src/3:374-398).  out[n_steps]. */
int hw1f_get_drift_table(const hw1f_engine* eng, int which, float sigma, float* out);
/* (int)(S1 / d_dt) exactly as the reference's fast-math build evaluates it on this GPU
 * (MUFU.RCP(d_dt)*S1 then F2I.TRUNC; common.cuh:322, src/3:46). */
int hw1f_steps_to(hw1f_engine* eng, float S1, int32_t* n_steps_S1);

/* ---- RNG handle ---------------------------------------------------------------- */
/* cudaMalloc(states) + init_rng<<<NB,NTPB>>>(states, seed)
 * (src/1:41,53; src/2:120,128,227,230; src/3:543,547,712,713; src/bench:94,95). */
int hw1f_rng_create(uint64_t seed, uint64_t first_path, uint64_t n_paths, hw1f_rng** out);
/* the state-array backup of src/3:407-409,494-497 (D2D copy of 48 B/path there) */
int hw1f_rng_clone(const hw1f_rng* src, hw1f_rng** out);
int hw1f_rng_destroy(hw1f_rng* rng);
/* number of normals every path has consumed so far (the reference keeps this implicitly
 * in the written-back curandState) */
int hw1f_rng_tell(const hw1f_rng* rng, uint64_t* normal_offset);
/* the state restore of src/3:422,434,502,509 */
int hw1f_rng_seek(hw1f_rng* rng, uint64_t normal_offset);
int hw1f_rng_info(const hw1f_rng* rng, uint64_t* seed, uint64_t* first_path, uint64_t* n_paths);
/* optional: build and cache the seed-independent jump tables for this handle's path range on `eng`
 * now (they are otherwise built by the first launch that needs them) */
int hw1f_rng_prepare(hw1f_engine* eng, const hw1f_rng* rng);

/* ---- Q1: zero-coupon curve -------------------------------------------------------- */
/* simulate_zcb<<<NB,NTPB>>> + compute_average_and_forward<<<1,128>>>
 * (include/market_data.cuh:25-127; src/1:65,75; src/3:471,474).
 * P[n_mat], f[n_mat]; P_se[n_mat] (standard error of P from the pair-sample variance; may be
 * NULL); sim_ms (CUDA-event time of the simulation, may be NULL).  Advances rng by n_steps. */
int hw1f_bond_curve(hw1f_engine* eng, hw1f_rng* rng, float* P, float* f, float* P_se, float* sim_ms);
/* The same call in two halves, for callers that loop over seeds or models (the reference's drivers do: 20 runs in
 * src/2:210-468 and src/3:527-654, one curve per bump in src/3:449-482): submit enqueues the jump-table launch, the
 * simulation and its tail and returns at once; the results land in result slot `slot` (mapped pinned host memory).
 * collect waits for that slot only and copies P, f (P_se may be NULL) out.  Up to HW1F_ASYNC_SLOTS submissions may be in
 * flight.  Every slot is a lane of its own: slot 0 runs on the engine's stream, slot k > 0 on an internal twin of the
 * engine (own stream, scratch and tables, created by the first submission to that slot; it follows every
 * hw1f_set_model / hw1f_engine_set_mode of the caller).  Walk the slots round robin and the GPU works on the next calls
 * -- jump tables, stream derivation of the first wave -- under the drain and the tail of the current one, while the host
 * reads the previous one.  Measured at 2^20 subsequences (tools/two_engine_probe.py, profiles/r02_submit_collect_lanes.txt):
 * 0.600 ms per call blocking, 0.564 / 0.558 / 0.553 with two / three / four slots in flight (0.580 when the calls in flight
 * shared one stream, i.e. without the overlap on the GPU).  Same kernels, same results bit for bit
 * as hw1f_bond_curve.  A slot must be collected before it is submitted to again; calls in different slots are not
 * ordered against each other; hw1f_engine_set_stream moves slot 0 only; hw1f_set_model with a different n_mat fails
 * while submissions are in flight; hw1f_bond_curve_ci refers to the last launch of slot 0 or of a blocking call (the other
 * lanes keep their block partials to themselves). */
#define HW1F_ASYNC_SLOTS 4
int hw1f_bond_curve_submit(hw1f_engine* eng, hw1f_rng* rng, int32_t slot);
int hw1f_bond_curve_collect(hw1f_engine* eng, int32_t slot, float* P, float* f, float* P_se);
/* split form: d_moments[2*n_mat] doubles on the device = {sum_m p0_m, sum_m p0_m^2} over this
 * handle's paths (entry 0 unused).  A caller may all-reduce d_moments across ranks before
 * calling hw1f_bond_curve_finish with the global path count. */
int hw1f_bond_curve_moments(hw1f_engine* eng, hw1f_rng* rng, double* d_moments);
int hw1f_bond_curve_finish(hw1f_engine* eng, const double* d_moments, uint64_t n_paths_total,
                           float* P, float* f, float* P_se);
/* Standard errors of f(0,T) and theta(T) for the LAST bond-curve launch on this engine (hw1f_bond_curve or
 * hw1f_bond_curve_moments; its per-block partial sums are still resident): covariance of P at neighbouring maturities
 * by batch means over the simulation blocks (independent batches of 1024 subsequences), then the delta method through
 * compute_average_and_forward (market_data.cuh:101-127) and recover_theta (src/2:14-35).  The reference reports no
 * interval for either; SURVEY 7.3-4 makes "inside the 95 % CI" the parity criterion for them.  Any output may be NULL;
 * P_se_batch is the batch-means standard error of P (cross-check of the exact P_se).  Needs >= 8 blocks. */
int hw1f_bond_curve_ci(hw1f_engine* eng, float* f_se, float* theta_se, float* P_se_batch);

/* ---- Q2a: theta calibration --------------------------------------------------------- */
/* recover_theta<<<1,N_MAT>>> (src/2_option_pricing.cu:14-35,82). All arrays [n_mat]. */
int hw1f_theta_calibrate(hw1f_engine* eng, const float* f, float* theta_rec, float* theta_ref, float* T);

/* ---- Q2b: ZBC with optimal-beta control variate ------------------------------------- */
typedef struct hw1f_zbc_result {
    double mom[5];          /* sum X, sum Y, sum X^2, sum Y^2, sum XY (per-thread pair sums, as the
                               reference accumulates them: common.cuh:356-362)          */
    uint64_t n_total;       /* 2 * n_paths                                             */
    int32_t n_steps_S1;
    int32_t reserved;
    /* float32 host algebra of src/2:154-179 and src/2:259-290, same operation order */
    float mean_X, mean_Y, var_X, var_Y, cov, beta, control_adjustment;
    float price_raw;        /* mean_X                                                  */
    float price_cv;         /* mean_X - beta (mean_Y - P0S2)                           */
    float corr_single;      /* "Correlation" of src/2:178 (algebraically beta)         */
    float corr;             /* rho of src/2:281                                        */
    /* additions (double algebra on the double moments) */
    double price_cv_f64, beta_f64, se_raw, se_cv, ci95_lo, ci95_hi;
    /* standard errors of beta* and rho from the five moments (the reference reports neither): regression slope,
     * sqrt((1 - rho^2) var_X / (var_Y (n - 2))), and Fisher's (1 - rho^2) / sqrt(n - 3), with ONE degree of freedom per
     * antithetic pair (the twins are dependent): n = n_total / 2 */
    double beta_se, corr_f64, corr_se;
} hw1f_zbc_result;

/* simulate_ZBC_control_variate<<<NB,NTPB>>> + host algebra (common.cuh:286-409; src/2:136,246;
 * src/3:127).  P_mkt/f_mkt[n_mat] as loaded from data/P.bin, data/f.bin.  n_steps_S1 < 0 derives
 * it with hw1f_steps_to.  Advances rng by n_steps_S1.  (Bumped-sigma pricing, i.e. what
 * run_finite_difference does around run_zbc_price, is hw1f_vega_fd below.) */
int hw1f_zbc_cv(hw1f_engine* eng, hw1f_rng* rng, float S1, float S2, float K,
                const float* P_mkt, const float* f_mkt, int32_t n_steps_S1,
                hw1f_zbc_result* out, float* sim_ms);
int hw1f_zbc_cv_moments(hw1f_engine* eng, hw1f_rng* rng, float S1, float S2, float K,
                        const float* P_mkt, const float* f_mkt, int32_t n_steps_S1, double* d_moments);
int hw1f_zbc_cv_finish(hw1f_engine* eng, const double* d_moments, uint64_t n_paths_total, float P0S2,
                       hw1f_zbc_result* out);
/* the 20-run validation of src/2:210-302 as ONE launch with a seed axis: seeds[n_runs] */
int hw1f_zbc_cv_batch(hw1f_engine* eng, const uint64_t* seeds, int32_t n_runs, uint64_t n_paths,
                      float S1, float S2, float K, const float* P_mkt, const float* f_mkt,
                      int32_t n_steps_S1, hw1f_zbc_result* out, float* sim_ms);

/* ---- Q3: vega ------------------------------------------------------------------------ */
typedef struct hw1f_vega_result {
    /* pathwise (simulate_sensitivity, src/3:22-96,251): sum / n_paths like src/3:261 */
    float vega_pathwise; double vega_pathwise_f64, vega_pathwise_se;
    /* finite differences with common random numbers (src/3:400-446) */
    float price_minus, price_plus, vega_fd;
    /* recalibrated FD (src/3:449-525) */
    float price_minus_recal, price_plus_recal, vega_fd_recal;
    int32_t n_steps_S1;
    float ms_pathwise, ms_fd, ms_fd_recal;
} hw1f_vega_result;

int hw1f_vega_pathwise(hw1f_engine* eng, hw1f_rng* rng, float S1, float S2, float K,
                       const float* P_mkt, const float* f_mkt, int32_t n_steps_S1,
                       hw1f_vega_result* out);
/* d_moments[2] = {sum v, sum v^2} */
int hw1f_vega_pathwise_moments(hw1f_engine* eng, hw1f_rng* rng, float S1, float S2, float K,
                               const float* P_mkt, const float* f_mkt, int32_t n_steps_S1, double* d_moments);
/* both bumps in ONE launch on the same normals (the reference restores a 50 MB state backup
 * between two launches, src/3:407-435).  Advances rng by n_steps_S1. */
int hw1f_vega_fd(hw1f_engine* eng, hw1f_rng* rng, float S1, float S2, float K,
                 const float* P_mkt, const float* f_mkt, float eps, int32_t n_steps_S1,
                 hw1f_vega_result* out);
/* recompute_market_data at sigma -/+ eps (both curves in one launch) then the two prices; the
 * handle is left where the reference leaves its state array (advanced by n_steps_S1).  The two
 * recalibrated curves are internal to the call (src/3:449-525 keeps them in device buffers that only
 * run_zbc_price reads): with S1 on the maturity grid the pass evaluates only the save points that
 * pricing interpolates on -- grid points around S1 and S2 and the last maturity -- same prices bit for bit. */
int hw1f_vega_fd_recalibrated(hw1f_engine* eng, hw1f_rng* rng, float S1, float S2, float K,
                              float eps, int32_t n_steps_S1, hw1f_vega_result* out);
/* the whole q3 sequence with the reference's draw windows: pathwise on normals [0,n),
 * FD-/+ on [n,2n), recalibrated curves on [2n,2n+N_STEPS) and prices on [2n,3n) (SURVEY 3.3) */
int hw1f_vega(hw1f_engine* eng, hw1f_rng* rng, float S1, float S2, float K,
              const float* P_mkt, const float* f_mkt, float eps, int32_t n_steps_S1,
              hw1f_vega_result* out);
/* the 20-run validation of src/3:527-568 as one launch with a seed axis; vega[n_runs] */
int hw1f_vega_pathwise_batch(hw1f_engine* eng, const uint64_t* seeds, int32_t n_runs, uint64_t n_paths,
                             float S1, float S2, float K, const float* P_mkt, const float* f_mkt,
                             int32_t n_steps_S1, float* vega, float* sim_ms);

/* ---- caps and floors: a strip of caplets in one simulation pass -------------------------- */
/* No reference call site: the reference prices one bond call (hw1f_zbc_cv).  A cap is a strip of zero-coupon bond PUTS,
 * a floor a strip of bond CALLS, one per reset date; one launch prices every caplet of the strip on one set of paths
 * (each path is stepped once to the last reset step and evaluated at every reset step on the way) and returns the
 * moments of each caplet and of the whole strip, in both arithmetic modes and at any normal offset.
 * The ABI speaks in bonds: a caplet on the rate L(T_r, T_p) with strike rate kappa, accrual tau and notional M equals
 * N ZBP(T_r, T_p, K) with K = 1 / (1 + tau kappa) and N = M (1 + tau kappa); a floorlet is the same with ZBC (the
 * Python layer's caplet_schedule() converts rates). */
typedef struct hw1f_caplet {
    float T_reset;          /* option expiry = reset date T_r (> 0)                                   */
    float T_pay;            /* bond maturity = payment date T_p, T_reset < T_pay <= T_final           */
    float K;                /* bond strike (> 0)                                                      */
    float N;                /* multiplier (> 0): payoff N (K - P)^+ for a cap, N (P - K)^+ for a floor */
    int32_t n_steps_reset;  /* step at which r is read; < 0: the step nearest to T_reset / dt          */
    int32_t reserved;
} hw1f_caplet;

/* Moments over antithetic PAIRS: X = x(+G) + x(-G), Y = y(+G) + y(-G) for each of the n_pairs = n_paths subsequences,
 * and every statistic is over the n_pairs samples of the pair means X/2, Y/2 (price_raw = sum X / (2 n_pairs),
 * se_raw = sqrt(var(X/2) / n_pairs)).  This differs from hw1f_zbc_result, whose second moments follow the reference
 * (per-twin sums, the twins treated as independent samples): these standard errors are honest. */
typedef struct hw1f_cap_result {   /* one caplet, or the whole strip */
    double mom[5];          /* sum X, sum Y, sum X^2, sum Y^2, sum XY over antithetic PAIRS: X = x(+G) + x(-G) */
    double price_raw, se_raw;
    double price_cv, se_cv; /* optimal-beta control variate, control Y = N D(T_r) P(T_r, T_p)             */
    double beta, corr;
    double control_mean;    /* known mean of the control: N P_mkt(T_p) interpolated like interp_mkt; summed for the strip */
} hw1f_cap_result;

#define HW1F_KIND_CAP 0
#define HW1F_KIND_FLOOR 1
#define HW1F_MAX_CAPLETS 100   /* 5 (100 + 1) = 505 doubles: fits the peer mailboxes (kCommMaxCount = 512) */

/* Reset steps ROUND to the nearest step (n_steps_reset < 0: lround(T_reset / dt) in double), unlike hw1f_steps_to, which
 * reproduces the reference's truncation for parity: a product date a hair below a step would otherwise move a reset by a
 * whole step.  HW1F_ERR_INVALID if |T_reset - k dt| > 1e-3 dt.
 * Every argument is checked before any launch; HW1F_ERR_INVALID (with a message) for: a kind other than HW1F_KIND_*,
 * n_caplets outside [1, HW1F_MAX_CAPLETS], reset steps that decrease along the strip or lie outside [1, n_steps],
 * T_pay <= T_reset or T_pay > T_final, K or N not finite and positive.  After a failure the rng has not moved and no
 * kernel was launched.
 * The strip's price uses ONE beta on Y_strip = sum_i Y_i; its price_raw is the sum of the caplets' up to rounding. */
/* out[n_caplets + 1]: the caplets in order, then the strip.  Advances rng by the last reset step. */
int hw1f_cap_floor(hw1f_engine* eng, hw1f_rng* rng, int32_t kind, const hw1f_caplet* caplets, int32_t n_caplets,
                   const float* P_mkt, const float* f_mkt, hw1f_cap_result* out, float* sim_ms);
/* split form, like every other estimator: d_moments[5 (n_caplets + 1)] on the device; honours hw1f_comm_attach */
int hw1f_cap_floor_moments(hw1f_engine* eng, hw1f_rng* rng, int32_t kind, const hw1f_caplet* caplets, int32_t n_caplets,
                           const float* P_mkt, const float* f_mkt, double* d_moments);
int hw1f_cap_floor_finish(hw1f_engine* eng, const double* d_moments, uint64_t n_paths_total, const hw1f_caplet* caplets,
                          int32_t n_caplets, const float* P_mkt, hw1f_cap_result* out);

/* ---- European swaptions: a book of coupon-bond options in one simulation pass ------------ */
/* No reference call site.  A coupon-bond option pays, at its exercise date T_e,
 *     N max(0, s (sum_j c_j P(T_e, T_j) - K)),   s = -1 payer (a put on the bond), +1 receiver (a call),
 * over its cash flows (T_j, c_j).  A swaption on a swap starting at T_e with fixed rate kappa, accruals tau_j and notional
 * M is the option with K = 1, c_j = kappa tau_j, c_last += 1 and N = M (the Python layer's swaption_schedule() builds
 * them).  One launch prices every option of the book on one set of paths, each read at its exercise step, and returns
 * the moments of each option and of the whole book, in both arithmetic modes and at any normal offset.  Payer and
 * receiver options may be mixed in one book. */
typedef struct hw1f_cash_flow {
    float T;                /* payment date, T_exercise < T <= T_final, strictly increasing within an option */
    float c;                /* amount per unit of N (> 0) */
} hw1f_cash_flow;

typedef struct hw1f_swaption {
    float T_exercise;       /* exercise date (> 0), on the step grid like T_reset of hw1f_caplet              */
    float K;                /* coupon-bond strike (> 0): 1 for a swap starting at T_exercise                   */
    float N;                /* multiplier (> 0)                                                                */
    int32_t kind;           /* HW1F_KIND_PAYER (put on the coupon bond) or HW1F_KIND_RECEIVER (call)          */
    int32_t n_steps_exercise;   /* step at which r is read; < 0: the step nearest to T_exercise / dt          */
    int32_t first_flow, n_flows;    /* this option's cash flows: flows[first_flow, first_flow + n_flows)     */
    int32_t reserved;
} hw1f_swaption;

#define HW1F_KIND_PAYER 0
#define HW1F_KIND_RECEIVER 1
#define HW1F_MAX_SWAPTIONS 100        /* 5 (100 + 1) = 505 doubles: fits the peer mailboxes, as for caps          */
#define HW1F_MAX_SWAPTION_FLOWS 2048  /* sum of n_flows over the book (a flow two options share counts twice):
                                       * the per-flow bond plans live in the kernel's shared memory                  */

/* Exercise steps round to the nearest step, as reset steps do for caplets.  The options must come in non-decreasing
 * exercise steps; several may share a step (an expiry x tenor grid).
 * Every argument is checked before any launch; HW1F_ERR_INVALID (with a message) for: a kind other than HW1F_KIND_PAYER /
 * HW1F_KIND_RECEIVER, n_swaptions outside [1, HW1F_MAX_SWAPTIONS], n_flows (the length of `flows`) < 1 or the sum of the
 * options' n_flows outside [1, HW1F_MAX_SWAPTION_FLOWS], an option's n_flows < 1 or a flow range outside `flows`, flow
 * dates not strictly increasing or with the first <= T_exercise or the last > T_final, c, K or N not finite and
 * positive (a forward-starting swap, whose first flow is negative, is out of scope), T_exercise off the step grid, an
 * exercise step outside [1, n_steps] or exercise steps that decrease along the book.  After a failure the rng has not
 * moved and no kernel was launched.
 * Moments and statistics follow hw1f_cap_result (antithetic pairs); the control of an option is
 * Y = N D(T_e) sum_j c_j P(T_e, T_j), whose known mean is N sum_j c_j P_mkt(T_j) (interpolated like interp_mkt).  The
 * book's price uses ONE beta on Y_book = sum_i Y_i. */
/* out[n_swaptions + 1]: the options in order, then the book.  Advances rng by the last exercise step. */
int hw1f_swaptions(hw1f_engine* eng, hw1f_rng* rng, const hw1f_swaption* swaptions, int32_t n_swaptions,
                   const hw1f_cash_flow* flows, int32_t n_flows, const float* P_mkt, const float* f_mkt,
                   hw1f_cap_result* out, float* sim_ms);
/* split form: d_moments[5 (n_swaptions + 1)] on the device; honours hw1f_comm_attach */
int hw1f_swaptions_moments(hw1f_engine* eng, hw1f_rng* rng, const hw1f_swaption* swaptions, int32_t n_swaptions,
                           const hw1f_cash_flow* flows, int32_t n_flows, const float* P_mkt, const float* f_mkt,
                           double* d_moments);
int hw1f_swaptions_finish(hw1f_engine* eng, const double* d_moments, uint64_t n_paths_total,
                          const hw1f_swaption* swaptions, int32_t n_swaptions, const hw1f_cash_flow* flows,
                          int32_t n_flows, const float* P_mkt, hw1f_cap_result* out);

/* ---- fused pass (BASELINE.json scaling run) --------------------------------------------- */
/* One launch: antithetic curve sums on the maturity grid + ZBC/control moments + pathwise-vega
 * tangent (both antithetic twins) evaluated at step n_steps_S1, all on the same normals.
 * d_moments layout: [0,2*n_mat) curve {sum p0, sum p0^2}; then the 5 ZBC moments; then
 * {sum (v1+v2), sum (v1+v2)^2, sum v1} with v1/v2 the pathwise vega sample of the +G/-G twin
 * (sum v1 equals hw1f_vega_pathwise_moments on the same handle position).  Advances rng by n_steps. */
#define HW1F_FUSED_EXTRA 8
int hw1f_fused_moments(hw1f_engine* eng, hw1f_rng* rng, float S1, float S2, float K,
                       const float* P_mkt, const float* f_mkt, int32_t n_steps_S1, double* d_moments);
/* the same pass with the two common-random-number FD bumps sigma -/+ eps of run_finite_difference
 * (src/3:400-446) riding on the same normals: d_moments gets HW1F_FUSED_FD_EXTRA more doubles
 * (5 ZBC moments at sigma-eps, 5 at sigma+eps) after the HW1F_FUSED_EXTRA block. */
#define HW1F_FUSED_FD_EXTRA 10
int hw1f_fused_fd_moments(hw1f_engine* eng, hw1f_rng* rng, float S1, float S2, float K,
                          const float* P_mkt, const float* f_mkt, float eps, int32_t n_steps_S1,
                          double* d_moments);
/* host-buffer form of the fused pass: ONE launch gives the curve (P, f, P_se), the ZBC price with
 * control variate (zbc), the antithetic pathwise vega and the CRN finite-difference vega (vega).
 * "Single-window" mode: every estimator reads normals [offset, offset+n_steps) -- statistically
 * equivalent to, but not stream-identical with, the reference's q3 (which uses a different draw
 * window per estimator; hw1f_vega reproduces those).  Advances rng by n_steps. */
int hw1f_fused(hw1f_engine* eng, hw1f_rng* rng, float S1, float S2, float K,
               const float* P_mkt, const float* f_mkt, float eps, int32_t n_steps_S1,
               float* P, float* f, float* P_se, hw1f_zbc_result* zbc, hw1f_vega_result* vega,
               float* sim_ms);

/* finalisation of a fused moment vector (after an optional all-reduce across ranks): the curve epilogue,
 * the ZBC algebra and the vegas from d_moments[2*n_mat + HW1F_FUSED_EXTRA (+ HW1F_FUSED_FD_EXTRA)].
 * eps > 0: the vector carries the FD block (hw1f_fused_fd_moments) and vega->price_minus/plus/vega_fd are
 * filled; eps <= 0: hw1f_fused_moments layout.  P0S2 = P_mkt[n_mat-1] of the market curve the pass used.
 * n_paths_total may exceed the reference's `int N_total` range (up to 2^40 subsequences: the scaling run);
 * the float32 algebra of src/2:154-179 then simply continues with (float)N_total. */
int hw1f_fused_finish(hw1f_engine* eng, const double* d_moments, uint64_t n_paths_total, float P0S2, float eps,
                      int32_t n_steps_S1, float* P, float* f, float* P_se, hw1f_zbc_result* zbc,
                      hw1f_vega_result* vega);

/* ---- single-process multi-GPU front end ------------------------------------------------------ */
/* One engine per device, paths sharded by contiguous XORWOW subsequence range (the union equals the
 * single-GPU path set bit for bit), ONE ncclAllReduce(ncclDouble, ncclSum) of the packed moment vector
 * per call, finalisation on device 0.  Nothing in the reference corresponds to this (it is single-GPU;
 * select_gpu() merely picks one device, common.cuh:122-141).  n_gpus <= 0 uses every visible device.
 * NCCL is dlopen'ed here; with one GPU no NCCL is needed. */
typedef struct hw1f_multi hw1f_multi;
int hw1f_multi_create(int n_gpus, hw1f_multi** out);
int hw1f_multi_destroy(hw1f_multi* m);
int hw1f_multi_device_count(const hw1f_multi* m, int* n_gpus);
const char* hw1f_multi_last_error(const hw1f_multi* m);
int hw1f_multi_set_model(hw1f_multi* m, const hw1f_params* p);
int hw1f_multi_set_mode(hw1f_multi* m, int mode);   /* HW1F_MODE_* on every device */
int hw1f_multi_bond_curve(hw1f_multi* m, uint64_t seed, uint64_t n_paths_total, uint64_t normal_offset,
                          float* P, float* f, float* P_se, float* wall_ms);
int hw1f_multi_zbc_cv(hw1f_multi* m, uint64_t seed, uint64_t n_paths_total, uint64_t normal_offset,
                      float S1, float S2, float K, const float* P_mkt, const float* f_mkt,
                      int32_t n_steps_S1, hw1f_zbc_result* out);
/* the BASELINE.json scaling run: hw1f_fused_fd_moments on every device's shard, one all-reduce of
 * 2*n_mat + 18 doubles, hw1f_fused_finish on device 0.  wall_ms: CUDA-event time on device 0 from the first
 * launch to the end of the all-reduce (may be NULL). */
int hw1f_multi_fused(hw1f_multi* m, uint64_t seed, uint64_t n_paths_total, uint64_t normal_offset, float S1, float S2,
                     float K, const float* P_mkt, const float* f_mkt, float eps, int32_t n_steps_S1, float* P,
                     float* f, float* P_se, hw1f_zbc_result* zbc, hw1f_vega_result* vega, float* wall_ms);
int hw1f_multi_vega_pathwise(hw1f_multi* m, uint64_t seed, uint64_t n_paths_total, uint64_t normal_offset,
                             float S1, float S2, float K, const float* P_mkt, const float* f_mkt,
                             int32_t n_steps_S1, double* vega, double* vega_se);

/* ---- peer-memory all-reduce (one process per GPU) ------------------------------------------------ */
/* The path's single exchange step -- summing the packed double moment vector over ranks -- as ONE own
 * kernel over NVLink peer memory instead of an NCCL call: every rank posts its vector into a mailbox
 * of every peer (CUDA IPC mapping), raises a system-scope flag, waits (bounded) for the peers' flags
 * and sums the slots in rank order, so the result is bit-identical on all ranks.  count <= 512, world <= 8.
 *   hw1f_comm_create : allocates this rank's mailbox, returns its 64-byte cudaIpcMemHandle_t
 *   (exchange the handles with any out-of-band all-gather, e.g. torch.distributed)
 *   hw1f_comm_connect: maps the peers' mailboxes; all_handles = world * 64 bytes in rank order;
 *                      cuda_stream = the stream the moments are produced on (engine stream)
 *   hw1f_comm_allreduce: enqueue; every rank must call it the same number of times
 *   hw1f_comm_timeouts: number of bounded-spin expiries so far (0 on a healthy run).  A timed-out call writes
 *                       NaN into d_data on that rank, and every *_finish call returns HW1F_ERR_COMM for a
 *                       non-finite moment vector: stale mailbox slots never turn into prices. */
typedef struct hw1f_comm hw1f_comm;
int hw1f_comm_create(hw1f_engine* eng, int world, void* ipc_handle64, hw1f_comm** out);
int hw1f_comm_connect(hw1f_comm* c, int rank, const void* all_handles, void* cuda_stream);
int hw1f_comm_allreduce(hw1f_comm* c, double* d_data, int32_t count);
/* on != 0: from now on every hw1f_*_moments entry point of the communicator's engine (bond curve, ZBC, pathwise, fused)
 * returns the ALL-REDUCED vector: the last block of the simulation kernel's reduction posts it to the peers and sums
 * the slots in rank order itself -- no launch between reduction and exchange.  Every rank must make the same calls in
 * the same order.  The one-call entry points (hw1f_bond_curve, hw1f_zbc_cv, ...) stay local.  on = 0 detaches. */
int hw1f_comm_attach(hw1f_comm* c, int on);
int hw1f_comm_timeouts(hw1f_comm* c, uint32_t* n);
int hw1f_comm_destroy(hw1f_comm* c);
const char* hw1f_comm_last_error(const hw1f_comm* c);

/* ---- sample trajectories -------------------------------------------------------------- */
/* simulate_paths_show<<<1,32>>> (market_data.cuh:136-160; src/1:163): r_paths[n_show*(n_steps+1)].
 * Does NOT advance rng (the reference's write-back is commented out, market_data.cuh:159). */
int hw1f_sample_paths(hw1f_engine* eng, const hw1f_rng* rng, int32_t n_show, float* r_paths);

/* ---- reduction benchmark ---------------------------------------------------------------- */
/* benchmark_kernel() of src/benchmark_reductions.cu:17-72 for one method:
 * 0 naive atomics, 1 shared-memory tree, 2 warp+block shuffle (perf_benchmark.cuh:19-197),
 * 3 the engine's deterministic two-level tree.  Advances rng by n_steps_S1 per launch. */
int hw1f_reduction_bench(hw1f_engine* eng, hw1f_rng* rng, int32_t method, float S1, float S2, float K,
                         const float* P_mkt, const float* f_mkt, int32_t n_steps_S1,
                         int32_t n_warmup, int32_t n_runs, float* avg_ms, float* price);

/* ---- introspection used by the parity tests ------------------------------------------------ */
/* raw XORWOW words derived ON THE GPU for path `path` of rng at its current offset:
 * state[6] = {d, v0..v4} then n_draws outputs of curand() */
int hw1f_debug_rng(hw1f_engine* eng, const hw1f_rng* rng, uint64_t path, int32_t n_draws,
                   uint32_t* state6, uint32_t* draws);
/* the first n normals of path `path` as the kernels generate them */
int hw1f_debug_normals(hw1f_engine* eng, const hw1f_rng* rng, uint64_t path, int32_t n, float* out);
/* HOST-side evaluation of the engine's jump algebra (no GPU): the XORWOW words after
 * curand_init(seed, path, 2*floor(normal_offset/2)): state6 = {d, v0..v4} */
int hw1f_host_rng_state(uint64_t seed, uint64_t path, uint64_t normal_offset, uint32_t* state6);
/* pipe-throughput micro-kernels that give the roofline denominators on this GPU: which =
 * 0 FFMA, 1 FFMA2, 2 MUFU.EX2, 3 SHF/LOP3, 4 I2FP.F32.U32, 5 MUFU+I2FP, 6 HW1F-like mix, 7 FMUL2,
 * 8 MUFU.LG2, 9 MUFU.SQRT, 10 MUFU.SIN, 11 MUFU.COS, 12 the Box-Muller MUFU mix (LG2, SQRT, SIN, COS in equal parts),
 * 13 that mix under the other instructions of the decomposed Q1 loop (the count is the MUFU instructions).
 * ms = event time of one launch, thread_instr = probed instructions executed (all threads). */
int hw1f_pipe_probe(hw1f_engine* eng, int32_t which, int32_t iters, float* ms, double* thread_instr);
/* number of kernel launches issued by this engine since creation */
int hw1f_launch_count(const hw1f_engine* eng, uint64_t* n);

#ifdef __cplusplus
}
#endif
#endif /* HW1F_H */
