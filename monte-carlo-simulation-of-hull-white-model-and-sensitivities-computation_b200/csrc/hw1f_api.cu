// hw1f_api.cu -- implementation of the C ABI declared in include/hw1f.h.
//
// Host side of the engine: model constants (host float32 arithmetic in the reference's order,
// common.cuh:60-110), per-device jump tables, launch orchestration on one CUDA stream, and the
// float32 estimator algebra of the reference drivers.  No CPU fallback exists: if a CUDA call
// fails the entry point returns an error code and hw1f_last_error() says why.
#include "../../include/hw1f.h"

#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <new>
#include <string>
#include <utility>
#include <vector>

#include "hw1f_kernels.cuh"
#include "hw1f_kernels_extra.cuh"
#include "hw1f_kernels_fast.cuh"
#include "hw1f_kernels_cap.cuh"
#include "hw1f_kernels_swaption.cuh"
#include "hw1f_tail.cuh"
#include "hw1f_probe.cuh"
#include "xorwow_jump.hpp"

using namespace hw1f;

// ---------------------------------------------------------------------------------------------
struct hw1f_rng {
    uint64_t seed, first_path, n_paths, offset;   // offset counted in normals
};

namespace {

constexpr int kTailCounters = 64;      // ticket counters of the tail kernel: one per run
constexpr int kSyncAreas = 4;          // result areas of the blocking entry points (mapped pinned host memory)
constexpr int kAsyncSlots = HW1F_ASYNC_SLOTS;   // + one area per submit / collect slot
constexpr int kResAreas = kSyncAreas + kAsyncSlots;

template <class T>
struct DevBuf {
    T* p = nullptr;
    size_t cap = 0;   // elements
    bool view = false;   // non-owning window into the model arena
    cudaError_t ensure(size_t n)
    {
        if (n <= cap) return cudaSuccess;
        if (view) return cudaErrorInvalidValue;
        if (p) cudaFree(p);
        p = nullptr;
        cap = 0;
        cudaError_t e = cudaMalloc(&p, n * sizeof(T));
        if (e == cudaSuccess) cap = n;
        return e;
    }
    void set_view(T* ptr, size_t n) { release(); p = ptr; cap = n; view = true; }
    void release() { if (p && !view) cudaFree(p); p = nullptr; cap = 0; view = false; }
};

struct Scenario {
    float sigma, sig_st;
    int drift_slot;    // which device drift table
};

}  // namespace

struct hw1f_engine {
    int device = -1;
    int sm_count = 148;
    size_t smem_optin = 0;
    cudaStream_t stream = nullptr, own_stream = nullptr;
    cudaEvent_t ev0 = nullptr, ev1 = nullptr, ev2 = nullptr, ev3 = nullptr, ev_stage = nullptr;
    cudaEvent_t ev_slot[HW1F_ASYNC_SLOTS] = {};   // hw1f_bond_curve_submit / _collect: one event per result slot
    bool slot_busy[HW1F_ASYNC_SLOTS] = {};
    // Every result slot is a lane of its own: slot 0 runs on this engine, slot k > 0 on a twin engine (own stream, scratch
    // and jump tables, created by the first submission to that slot, same model and mode), so that submissions in flight
    // overlap on the GPU -- the jump-table launch and the first wave's stream derivation of one call run under the drain
    // and the tail of another
    hw1f_engine* twin[HW1F_ASYNC_SLOTS] = {};   // [0] unused
    uint64_t model_gen = 0, twin_gen[HW1F_ASYNC_SLOTS] = {};   // hw1f_set_model calls seen by this engine / forwarded to a twin
    std::string err = "";
    uint64_t launches = 0;

    int mode = HW1F_MODE_DECOMPOSED;
    bool has_model = false;
    hw1f_params p{};
    float dt = 0, spacing = 0, exp_adt = 0, sig_st = 0;
    int stride = 0;
    std::vector<float> h_drift, h_sdrift;

    DevBuf<uint32_t> d_Jpow2;            // [kNumPow][800]
    DevBuf<uint32_t> d_Jnib;             // [4][16][800]: J^(n 16^j), the nibble powers prep_lo_kernel applies
    DevBuf<uint32_t> d_W;                // window tables of the high jump matrices: [four-bit | five-bit] per matrix
    uint32_t W_hi_base = 0, W_n_hi = 0, W_L_log2 = 0;
    DevBuf<uint32_t> d_U;                // [n_runs][5][L]
    // drift tables, duplicated float2: slot 0 base, 1 sensitivity, 2/3 bumped scenarios
    DevBuf<float2> d_drift[4];
    DevBuf<float> d_mkt;                 // [4][n_mat]: P0,f0,P1,f1
    DevBuf<float> d_center;              // [n_mat] centring constants of the curve accumulation
    // noise-free ("deterministic") parts per drift slot, host double: det_m[slot][i] = short rate
    // after i steps with G = 0, det_I[slot][i] its trapezoid integral (slot 1: tangent D, ID)
    std::vector<double> det_m[4], det_I[4];
    DevBuf<float> d_emI[4];              // [n_mat] exp(-det_I) at the save points (decomposed curve kernels)
    DevBuf<BondPlan> d_plans;
    DevBuf<double> d_partials;
    DevBuf<float2> d_state;              // dumped noise state (h, q) per subsequence (recalibrated FD, one pass)
    DevBuf<double> d_moments;            // internal moment vector
    DevBuf<float> d_out;                 // epilogue outputs
    DevBuf<char> d_cap;                  // hw1f_cap_floor* / hw1f_swaptions*: product tables + market curves, one staged upload per call
    DevBuf<int> d_int;
    void* h_stage = nullptr;             // pinned
    size_t h_stage_bytes = 0;
    // model arena: base drift, sensitivity drift, centring constants and exp(-Im) in ONE device
    // allocation with a pinned host mirror, so set_model is a single H2D copy (tables are rebuilt
    // only when the parameters change)
    DevBuf<char> d_model;
    char* h_model = nullptr;
    size_t model_bytes = 0, model_off_emI = 0;
    bool model_cached = false;
    hw1f_params cached_p{};
    // FD arena: shifted drift tables and exp(-Im) of the sigma -/+ eps scenarios (slots 2, 3) in one device
    // allocation with a pinned host mirror; rebuilt on the host only when (model, sigma pair) changes,
    // uploaded with ONE copy per pricing call (the reference re-sends the tables per bump, src/3:416-441)
    DevBuf<char> d_fd;
    char* h_fd = nullptr;
    size_t fd_bytes = 0;
    bool fd_cached = false;
    float fd_sig[2] = {0.f, 0.f};
    cudaEvent_t ev_fd = nullptr;
    // tail of the simulation kernels (hw1f_tail.cuh): ticket counters, group partials, and the result areas in mapped
    // pinned host memory the last block stores into (the host only waits for the stream)
    DevBuf<unsigned> d_tail_cnt;
    DevBuf<double> d_gpart;
    char* h_res = nullptr;
    size_t res_area_bytes = 0, res_doubles = 0;
    // the last single-scenario bond-curve launch whose block partials are still in d_partials (hw1f_bond_curve_ci)
    bool seq_one_launch = true;          // hw1f_vega: the whole Q3 sequence as one simulation launch (HW1F_Q3_ONE_LAUNCH=0 disables)
    bool ci_valid = false;
    StreamGeom ci_geom{};
    unsigned ci_blocks = 0;
    // peers attached with hw1f_comm_attach: the *_moments entry points all-reduce in their tail
    bool comm_on = false;
    CommDev comm{};
    unsigned* comm_epoch = nullptr;
    // (int)(S1/d_dt) as the device evaluates it (hw1f_steps_to): one probe per (S1, dt)
    bool steps_cached = false;
    float steps_S1 = 0.f, steps_dt = 0.f;
    int32_t steps_n = 0;
};

namespace {

#define HW_CUDA(eng, call)                                                                       \
    do {                                                                                         \
        cudaError_t _e = (call);                                                                 \
        if (_e != cudaSuccess) {                                                                 \
            (eng)->err = std::string(#call) + ": " + cudaGetErrorString(_e);                     \
            return HW1F_ERR_CUDA;                                                                \
        }                                                                                        \
    } while (0)

#define HW_REQUIRE(eng, cond, msg)                                                               \
    do {                                                                                         \
        if (!(cond)) { (eng)->err = (msg); return HW1F_ERR_INVALID; }                            \
    } while (0)

#define HW_TRY(expr)                                                                             \
    do { int _s = (expr); if (_s != HW1F_OK) return _s; } while (0)

int check_launch(hw1f_engine* e, const char* what)
{
    cudaError_t err = cudaGetLastError();
    ++e->launches;
    if (err != cudaSuccess) {
        e->err = std::string(what) + ": " + cudaGetErrorString(err);
        return HW1F_ERR_CUDA;
    }
    return HW1F_OK;
}

// ---- host model constants: the reference's host float32 expressions -------------------------
void host_drift_tables(const hw1f_params& p, float sigma, float* drift, float* sdrift)
{
    // compute_drift_tables, common.cuh:60-84
    const float H_A = p.a, H_DT = p.T_final / p.n_steps;
    const float h_exp_adt = expf(-H_A * H_DT);
    const float om_a = (1.0f - h_exp_adt) / H_A;
    const float om_a_sq = om_a / H_A;
    for (int i = 0; i < p.n_steps; ++i) {
        const float s = i * H_DT;
        const float t = (i + 1) * H_DT;
        const float first_term = ((s + H_DT) - h_exp_adt * s) / H_A - om_a_sq;
        if (drift)
            drift[i] = (s < p.theta_break) ? (p.theta_b0 * first_term + p.theta_a0 * om_a)
                                           : (p.theta_b1 * first_term + p.theta_a1 * om_a);
        if (sdrift) {
            const float sigma_term = (2.0f * sigma * expf(-H_A * t)) * (coshf(H_A * t) - coshf(H_A * s));
            sdrift[i] = sigma_term / (H_A * H_A);
        }
    }
}

void host_shifted_drift_table(const hw1f_params& p, float sigma_new, float sigma_old, float* out)
{
    // compute_shifted_drift_table, src/3_sensitivity_analysis.cu:374-398
    const float H_A = p.a, H_DT = p.T_final / p.n_steps;
    const float shift_coeff = (sigma_new * sigma_new - sigma_old * sigma_old) / (2.0f * H_A);
    const float h_exp_adt = expf(-H_A * H_DT);
    const float om_a = (1.0f - h_exp_adt) / H_A;
    const float om_a_sq = om_a / H_A;
    for (int i = 0; i < p.n_steps; ++i) {
        const float s = i * H_DT;
        const float t = (i + 1) * H_DT;
        const float first_term = ((s + H_DT) - h_exp_adt * s) / H_A - om_a_sq;
        const float base = (s < p.theta_break) ? (p.theta_b0 * first_term + p.theta_a0 * om_a)
                                               : (p.theta_b1 * first_term + p.fd_theta_a1 * om_a);
        const float adj = (shift_coeff / H_A) *
                          (1.0f + expf(-2.0f * H_A * t) - expf(-H_A * (t - s)) - expf(-H_A * (t + s)));
        out[i] = base + adj;
    }
}

float host_sig_st(const hw1f_params& p, float sigma)
{
    // compute_h_sig_st, common.cuh:87-89
    const float H_DT = p.T_final / p.n_steps;
    return sigma * sqrtf((1.0f - expf(-2.0f * p.a * H_DT)) / (2.0f * p.a));
}

// ---- staging ---------------------------------------------------------------------------------
int stage_reserve(hw1f_engine* e, size_t bytes)
{
    if (bytes <= e->h_stage_bytes) return HW1F_OK;
    if (e->h_stage) cudaFreeHost(e->h_stage);
    e->h_stage = nullptr;
    e->h_stage_bytes = 0;
    HW_CUDA(e, cudaMallocHost(&e->h_stage, bytes));
    e->h_stage_bytes = bytes;
    return HW1F_OK;
}

// host -> device through the pinned buffer, stream ordered; waits for the previous upload only
int upload(hw1f_engine* e, void* dst, const void* src, size_t bytes)
{
    HW_CUDA(e, cudaEventSynchronize(e->ev_stage));
    HW_TRY(stage_reserve(e, bytes));
    memcpy(e->h_stage, src, bytes);
    HW_CUDA(e, cudaMemcpyAsync(dst, e->h_stage, bytes, cudaMemcpyHostToDevice, e->stream));
    HW_CUDA(e, cudaEventRecord(e->ev_stage, e->stream));
    return HW1F_OK;
}

// device -> host through the pinned buffer; synchronises the stream
int download(hw1f_engine* e, void* dst, const void* src, size_t bytes)
{
    HW_CUDA(e, cudaEventSynchronize(e->ev_stage));
    HW_TRY(stage_reserve(e, bytes));
    HW_CUDA(e, cudaMemcpyAsync(e->h_stage, src, bytes, cudaMemcpyDeviceToHost, e->stream));
    HW_CUDA(e, cudaStreamSynchronize(e->stream));
    memcpy(dst, e->h_stage, bytes);
    return HW1F_OK;
}

// noise-free recursion with a drift table (start r0 for rate tables, 0 for the tangent table);
// fills det_m/det_I[slot] and, for rate tables, emI[n_mat] = exp(-Im) at the save points
void build_det_tables(hw1f_engine* e, int slot, const float* table, float* emI)
{
    const int n = e->p.n_steps, nm = e->p.n_mat;
    std::vector<double>& m = e->det_m[slot];
    std::vector<double>& I = e->det_I[slot];
    m.assign(n + 1, 0.0);
    I.assign(n + 1, 0.0);
    m[0] = (slot == 1) ? 0.0 : (double)e->p.r0;
    for (int i = 0; i < n; ++i) {
        m[i + 1] = m[i] * (double)e->exp_adt + (double)table[i];
        I[i + 1] = I[i] + 0.5 * (m[i] + m[i + 1]) * (double)e->dt;
    }
    if (emI) {
        emI[0] = 1.0f;
        for (int k = 1; k < nm; ++k) emI[k] = (float)exp(-I[(size_t)k * e->stride]);
    }
}

// bumped-sigma scenario tables (slots 2, 3) of run_finite_difference (src/3:400-446): shifted drift tables
// (duplicated float2) and exp(-Im) of sigma -/+ eps.  Host-side construction is cached per (model, sigma
// pair); every call sends the arena with one stream-ordered copy.
int upload_fd_tables(hw1f_engine* e, float sig_m, float sig_p)
{
    const int n = e->p.n_steps, nm = e->p.n_mat;
    auto align = [](size_t x) { return (x + 255) & ~(size_t)255; };
    const size_t sz_d = align((size_t)(n + 2) * sizeof(float2)), sz_e = align((size_t)nm * sizeof(float));
    const size_t total = 2 * sz_d + 2 * sz_e;
    if (total != e->fd_bytes) {
        HW_CUDA(e, cudaStreamSynchronize(e->stream));
        e->d_drift[2].release(); e->d_drift[3].release(); e->d_emI[2].release(); e->d_emI[3].release();
        e->d_fd.release();
        if (e->h_fd) cudaFreeHost(e->h_fd);
        e->h_fd = nullptr;
        e->fd_bytes = 0;
        e->fd_cached = false;
        HW_CUDA(e, e->d_fd.ensure(total));
        HW_CUDA(e, cudaMallocHost((void**)&e->h_fd, total));
        e->fd_bytes = total;
        e->d_drift[2].set_view(reinterpret_cast<float2*>(e->d_fd.p), n + 2);
        e->d_drift[3].set_view(reinterpret_cast<float2*>(e->d_fd.p + sz_d), n + 2);
        e->d_emI[2].set_view(reinterpret_cast<float*>(e->d_fd.p + 2 * sz_d), nm);
        e->d_emI[3].set_view(reinterpret_cast<float*>(e->d_fd.p + 2 * sz_d + sz_e), nm);
    }
    if (!(e->fd_cached && e->fd_sig[0] == sig_m && e->fd_sig[1] == sig_p)) {
        HW_CUDA(e, cudaEventSynchronize(e->ev_fd));   // a previous upload may still read the pinned mirror
        memset(e->h_fd, 0, total);
        std::vector<float> tab(n);
        for (int k = 0; k < 2; ++k) {
            host_shifted_drift_table(e->p, k ? sig_p : sig_m, e->p.sigma, tab.data());
            float2* dup = reinterpret_cast<float2*>(e->h_fd + k * sz_d);
            for (int i = 0; i < n; ++i) dup[i] = make_float2(tab[i], tab[i]);
            build_det_tables(e, 2 + k, tab.data(), reinterpret_cast<float*>(e->h_fd + 2 * sz_d + k * sz_e));
        }
        e->fd_sig[0] = sig_m;
        e->fd_sig[1] = sig_p;
        e->fd_cached = true;
    }
    HW_CUDA(e, cudaMemcpyAsync(e->d_fd.p, e->h_fd, total, cudaMemcpyHostToDevice, e->stream));
    HW_CUDA(e, cudaEventRecord(e->ev_fd, e->stream));
    return HW1F_OK;
}

ModelDev model_dev(const hw1f_engine* e)
{
    ModelDev m;
    m.r0 = e->p.r0;
    m.exp_adt = e->exp_adt;
    m.exp_2adt = e->exp_adt * e->exp_adt;
    {
        const double ed = (double)e->exp_adt, rho = (ed * ed - (double)m.exp_2adt) / (double)m.exp_2adt;
        m.rho1 = (float)rho;
        m.rho5 = (float)(5.0 * rho);
        m.qA = (float)(2.0 / (1.0 - ed));
        m.qB = (float)(2.0 * ed / (1.0 - ed) + 1.0);
    }
    m.dt = e->dt;
    m.a = e->p.a;
    m.spacing = e->spacing;
    m.inv_spacing = 1.0f / e->spacing;   // the compiler folds x/0.1f to x*10.0f in the reference
    m.neg_spacing = -e->spacing;
    m.n_steps = e->p.n_steps;
    m.n_mat = e->p.n_mat;
    m.stride = e->stride;
    return m;
}

// ---- stream geometry: window tables for the hi part, U table for the lo part -------------------
struct Launch {
    StreamGeom g;
    SeedArgs seeds;
    int n_runs;
    unsigned grid_x;
    int lead;          // 1 if the launch starts on the cos half of a Box-Muller pair
};

uint32_t pick_L_log2(uint64_t n_paths)
{
    uint32_t lg = 0;
    while ((1ull << lg) < n_paths) ++lg;
    static const int bias = std::getenv("HW1F_L_BIAS") ? std::atoi(std::getenv("HW1F_L_BIAS")) : 0;   // A/B only
    uint32_t L = lg / 2 + 1 + bias;
    if (L < (uint32_t)kChunkLog2) L = kChunkLog2;
    if (L > 16) L = 16;
    return L;
}

int ensure_tables(hw1f_engine* e)
{
    if (e->d_Jpow2.p) return HW1F_OK;
    const std::vector<uint32_t> flat = jump_tables().flat_seq();
    HW_CUDA(e, e->d_Jpow2.ensure(flat.size()));
    HW_CUDA(e, cudaMemcpyAsync(e->d_Jpow2.p, flat.data(), flat.size() * sizeof(uint32_t), cudaMemcpyHostToDevice,
                               e->stream));
    const std::vector<uint32_t> nib = jump_tables().flat_seq_nibbles();
    HW_CUDA(e, e->d_Jnib.ensure(nib.size()));
    HW_CUDA(e, cudaMemcpyAsync(e->d_Jnib.p, nib.data(), nib.size() * sizeof(uint32_t), cudaMemcpyHostToDevice, e->stream));
    HW_CUDA(e, cudaStreamSynchronize(e->stream));
    return HW1F_OK;
}

int ensure_windows(hw1f_engine* e, uint32_t L_log2, uint32_t hi_first, uint32_t hi_last)
{
    if (e->d_W.p && e->W_L_log2 == L_log2 && hi_first >= e->W_hi_base && hi_last < e->W_hi_base + e->W_n_hi)
        return HW1F_OK;
    const uint32_t n_hi = hi_last - hi_first + 1;
    HW_CUDA(e, e->d_W.ensure((size_t)n_hi * kWinStride));
    build_hi_kernel<<<n_hi, 160, 0, e->stream>>>(hi_first, L_log2, e->d_Jpow2.p, e->d_W.p);
    HW_TRY(check_launch(e, "build_hi_kernel"));
    e->W_L_log2 = L_log2;
    e->W_hi_base = hi_first;
    e->W_n_hi = n_hi;
    return HW1F_OK;
}

ModelDev model_dev(const hw1f_engine* e);

// a launch with (or without) programmatic stream serialisation: the simulation kernels start while the prep_lo_kernel
// in front of them is still running and wait for it with griddepcontrol.wait (hw1f_kernels_fast.cuh)
template <class... KArgs, class... Args>
cudaError_t launch_k(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t stream, bool pdl,
                     Args&&... args)
{
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = grid;
    cfg.blockDim = block;
    cfg.dynamicSmemBytes = smem;
    cfg.stream = stream;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = pdl ? 1 : 0;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    return cudaLaunchKernelEx(&cfg, kernel, KArgs(std::forward<Args>(args))...);
}

// Prepare a launch over `n_runs` seeds sharing (first_path, n_paths, normal offset).  `job` (optional): bond plans
// computed by an extra block of the same prep_lo_kernel launch.
int prepare_launch(hw1f_engine* e, const uint64_t* seeds, int n_runs, uint64_t first_path, uint64_t n_paths,
                   uint64_t normal_offset, Launch* L, const PlanJob* job = nullptr)
{
    HW_REQUIRE(e, n_runs >= 1 && n_runs <= kMaxRuns, "n_runs must be in [1,32]");
    HW_REQUIRE(e, n_paths >= 1, "n_paths must be >= 1");
    e->ci_valid = false;   // the launch that follows overwrites the block partials
    HW_REQUIRE(e, first_path + n_paths >= first_path, "path range overflows 64 bits");
    HW_TRY(ensure_tables(e));
    const uint32_t L_log2 = pick_L_log2(n_paths);
    const uint64_t last_path = first_path + n_paths - 1;
    const uint64_t hi_first = first_path >> L_log2, hi_last = last_path >> L_log2;
    HW_REQUIRE(e, hi_last < (1ull << 32), "path index too large for the jump tables (>= 2^41)");
    HW_TRY(ensure_windows(e, L_log2, (uint32_t)hi_first, (uint32_t)hi_last));
    const uint32_t Lsz = 1u << L_log2;
    HW_CUDA(e, e->d_U.ensure((size_t)n_runs * 5 * Lsz));

    // seed scramble + offset jump on the host (one 160-bit vector per run)
    const uint64_t draw_offset = 2 * (normal_offset / 2);
    const JumpTables& jt = jump_tables();
    for (int r = 0; r < n_runs; ++r) {
        BitVec v;
        const uint32_t d0 = seed_scramble(seeds[r], v);
        uint64_t off = draw_offset;
        for (int k = 0; off != 0 && k < kNumPow; ++k, off >>= 1)
            if (off & 1) v = jt.step_pow2[k].apply(v);
        HW_REQUIRE(e, off == 0, "normal offset too large (>= 2^48)");
        for (int w = 0; w < 5; ++w) L->seeds.s[r].v0[w] = v[w];
        L->seeds.s[r].d_start = d0 + kWeyl * (uint32_t)draw_offset;
    }
    for (int r = n_runs; r < kMaxRuns; ++r) L->seeds.s[r] = L->seeds.s[0];
    L->n_runs = n_runs;
    L->lead = (int)(normal_offset & 1);

    const unsigned long long total_warps = (unsigned long long)n_runs * Lsz;
    const unsigned prep_blocks = (unsigned)((total_warps + 7) / 8);
    PlanJob no_job{};
    if (job) HW_CUDA(e, e->d_plans.ensure(4));
    // + 1: the plan block
    prep_lo_kernel<<<prep_blocks + 1, 256, 0, e->stream>>>(L->seeds, n_runs, L_log2, e->d_Jnib.p, e->d_U.p, model_dev(e),
                                                          job ? *job : no_job);
    HW_TRY(check_launch(e, "prep_lo_kernel"));

    StreamGeom& g = L->g;
    g.W = e->d_W.p;
    g.U = e->d_U.p;
    g.first_path = first_path;
    g.n_paths = n_paths;
    g.chunk0 = first_path >> kChunkLog2;
    g.n_chunks = (last_path >> kChunkLog2) - g.chunk0 + 1;
    g.hi_base = e->W_hi_base;
    g.L_log2 = L_log2;
    // one wave of resident blocks per grid-stride pass keeps the partials small at 2^30 paths
    const unsigned long long cap = (unsigned long long)e->sm_count * 32ull;
    L->grid_x = (unsigned)(g.n_chunks < cap ? g.n_chunks : cap);
    return HW1F_OK;
}

// sums `count` entries starting at `offset` of partials[run][block][stride] into d_out[run*out_stride + ..]
int reduce_range(hw1f_engine* e, int n_runs, unsigned n_blocks, int stride, int offset, int count, double* d_out,
                 int out_stride)
{
    if (count <= 0) return HW1F_OK;
    reduce_partials_kernel<double><<<dim3(count, n_runs), 256, 0, e->stream>>>(e->d_partials.p + offset, (int)n_blocks,
                                                                             stride, d_out, out_stride);
    return check_launch(e, "reduce_partials_kernel");
}

int reduce_to(hw1f_engine* e, int n_runs, unsigned n_blocks, int nq, double* d_out)
{
    return reduce_range(e, n_runs, n_blocks, nq, 0, nq, d_out, nq);
}

int require_model(hw1f_engine* e)
{
    if (!e) return HW1F_ERR_INVALID;
    if (!e->has_model) { e->err = "hw1f_set_model() has not been called"; return HW1F_ERR_NO_MODEL; }
    return HW1F_OK;
}

int resolve_steps(hw1f_engine* e, float S1, int32_t n_in, int32_t* n_out)
{
    if (n_in >= 0) { *n_out = n_in; }
    else HW_TRY(hw1f_steps_to(e, S1, n_out));
    HW_REQUIRE(e, *n_out >= 0 && *n_out <= e->p.n_steps, "n_steps_S1 outside [0, n_steps]");
    return HW1F_OK;
}

// ---- bond plans: path-independent part of P(S1,S2), computed on the device as a side job --------
// plans for up to three scenarios priced on HOST-resident market curves: the six values a plan reads travel as kernel
// arguments (no market upload).  Plans go to d_plans[slot0 ..).
PlanJob plan_job_host(hw1f_engine* e, const ScenDev* sc, int n_scen, float S1, float S2, const float* P_mkt,
                      const float* f_mkt, int slot0 = 0)
{
    const int n = e->p.n_mat;
    const ModelDev md = model_dev(e);
    PlanJob job{};
    auto pick = [&](const float* data, float T, float out[2]) {
        const float prod = T * md.inv_spacing;           // IEEE single multiply, like mul_() on the device
        int idx = (prod >= (float)n) ? n : (int)prod;    // (int): truncation = __float2int_rz
        if (idx < 0) idx = 0;
        if (idx >= n - 1) { out[0] = data[n - 1]; out[1] = data[n - 1]; }
        else { out[0] = data[idx]; out[1] = data[idx + 1]; }
        return idx;
    };
    job.pts.idx_S2 = pick(P_mkt, S2, job.pts.P_S2);
    job.pts.idx_S1 = pick(P_mkt, S1, job.pts.P_S1);
    pick(f_mkt, S1, job.pts.f_S1);
    job.use_pts = 1;
    job.n_scen = n_scen;
    for (int s = 0; s < n_scen; ++s) { job.sigma[s] = sc[s].sigma; job.sig_st[s] = sc[s].sig_st; }
    job.S1 = S1;
    job.S2 = S2;
    job.plans = e->d_plans.p + slot0;   // d_plans holds 4 entries from engine creation on
    return job;
}

// plans for two scenarios on DEVICE-resident market curves (the recalibrated FD's own curves): market set s at
// d_mkt[2s], d_mkt[2s+1]
PlanJob plan_job_dev(hw1f_engine* e, const ScenDev* sc, int n_scen, float S1, float S2)
{
    const int n = e->p.n_mat;
    PlanJob job{};
    job.n_scen = n_scen;
    for (int s = 0; s < n_scen; ++s) { job.sigma[s] = sc[s].sigma; job.sig_st[s] = sc[s].sig_st; }
    job.S1 = S1;
    job.S2 = S2;
    job.use_pts = 0;
    for (int s = 0; s < 2; ++s) {
        job.P_mkt[s] = e->d_mkt.p + 2 * (size_t)(n_scen > 1 ? s : 0) * n;
        job.f_mkt[s] = job.P_mkt[s] + n;
    }
    job.plans = e->d_plans.p;
    return job;
}

// Save points a recalibration-curve pass (fast_kernel DUMP) has to evaluate: the pricing behind it interpolates P and f
// at S1 and P at S2 on the grid (compute_plan: data[idx], data[idx + 1]; f[m] differences P[m -+ 1]) and reads P at the
// last maturity (P(0,S2) of run_zbc_price, src/3:140-157).  Two windows of six grid points from idx - 2 on; the kernel
// adds the last two grid points.  Bit 31 marks the code (lead >= 0: every save point).
int keep_code(const hw1f_engine* e, float S1, float S2)
{
    const int n = e->p.n_mat;
    const float inv = 1.0f / e->spacing;
    auto first = [&](float T) {
        const float prod = T * inv;
        int idx = (prod >= (float)n) ? n : (int)prod;
        idx -= 2;
        if (idx < 0) idx = 0;
        if (idx > 1023) idx = 1023;
        return (unsigned)idx;
    };
    return (int)(first(S1) | (first(S2) << 10) | 0x80000000u);
}

int launch_plan_job(hw1f_engine* e, const PlanJob& job)
{
    plan_job_kernel<<<1, 32, 0, e->stream>>>(model_dev(e), job);
    return check_launch(e, "plan_job_kernel");
}

ScenDev scen_dev(const hw1f_engine* e, float sigma, float sig_st, int drift_slot)
{
    ScenDev s;
    s.sigma = sigma;
    s.sig_st = sig_st;
    s.drift2 = e->d_drift[drift_slot].p;
    s.sdrift2 = e->d_drift[1].p;
    s.center = e->d_center.p;
    s.slot = drift_slot;
    return s;
}

// decomposed-mode constants of one sigma scenario (drift slot selects the noise-free tables)
FastScen fast_scen(const hw1f_engine* e, float sig_st, int drift_slot, int n_steps_S1)
{
    FastScen f;
    f.sg = sig_st;
    f.c = (0.5f * e->dt) * sig_st;
    f.mS1 = (float)e->det_m[drift_slot][n_steps_S1];
    f.ImS1 = (float)e->det_I[drift_slot][n_steps_S1];
    f.emI = e->d_emI[drift_slot].p;
    return f;
}

FastTangent fast_tangent(const hw1f_engine* e, int n_steps_S1)
{
    FastTangent t;
    t.DS1 = (float)e->det_m[1][n_steps_S1];
    t.IDS1 = (float)e->det_I[1][n_steps_S1];
    return t;
}

int drift_slot_of(const hw1f_engine*, const ScenDev& sc) { return sc.slot; }

// (ncur, nzbc, pw, seq): the template arguments of the fast_kernel instantiation (they pick the window table it stages)
size_t smem_fast(const hw1f_engine* e, int ncur, int nzbc, int pw, int seq = 0)
{
    const size_t nqc = (size_t)ncur * 2 * e->p.n_mat;
    return (size_t)fast_win_words(ncur, nzbc, pw, seq) * 4 + nqc * sizeof(double) + (size_t)kWarps * nqc * sizeof(float) +
           (size_t)ncur * e->p.n_mat * sizeof(float) + 64;
}

size_t smem_curve(const hw1f_engine* e, int nscen)
{
    const int nq = nscen * 2 * e->p.n_mat;
    return (size_t)kWinWords * 4 + (size_t)nscen * ((e->p.n_steps + 1) / 2) * sizeof(float4) + (size_t)nq * sizeof(double) +
           (size_t)kWarps * nq * sizeof(float) + (size_t)nscen * e->p.n_mat * sizeof(float);
}

// dynamic shared memory: every simulation kernel is opted in to the device maximum ONCE at engine
// creation (init_kernels); per launch only the requested size is checked
template <class K>
int set_smem(hw1f_engine* e, K, size_t bytes)
{
    if (bytes + 2048 > e->smem_optin) {   // 2 KB head-room for the kernels' static shared arrays
        e->err = "model too large for shared memory (n_mat or n_steps x scenarios of this pass; see the size limits in hw1f.h)";
        return HW1F_ERR_UNSUPPORTED;
    }
    return HW1F_OK;
}

template <class K>
cudaError_t opt_in(K kernel, size_t bytes)
{
    cudaFuncAttributes attr;
    cudaError_t err = cudaFuncGetAttributes(&attr, kernel);   // also forces the module load
    if (err != cudaSuccess) return err;
    if (bytes > attr.sharedSizeBytes) bytes -= attr.sharedSizeBytes;   // static + dynamic <= opt-in limit
    err = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);
    if (err != cudaSuccess) return err;
    return cudaFuncSetAttribute(kernel, cudaFuncAttributePreferredSharedMemoryCarveout, (int)cudaSharedmemCarveoutMaxShared);
}

// ---- what happens after the block partials exist (hw1f_tail.cuh) ---------------------------------
// Finish says what the last block of a simulation launch does beyond storing the device moment vector; in
// reference-order mode (separate reduction kernels) the same steps run as tail_publish_kernel.
struct Finish {
    double* host_mom = nullptr;     // copy of the moment vector in mapped pinned host memory
    bool exchange = false;          // all-reduce with the attached peers (hw1f_comm_attach)
    bool epi = false;               // curve epilogue: P, f (P_se) of every curve scenario
    uint64_t n_total = 0;           //   subsequences over all ranks
    float* dev_curve = nullptr;     //   [ncur][2][n_mat] on the device
    float* host_curve = nullptr;    //   [ncur][3][n_mat] in mapped pinned host memory
    PlanJob plan{};                 // bond plans on dev_curve afterwards
};

// result areas in mapped pinned host memory: area k = [res_doubles doubles][res_floats floats]
double* res_mom(const hw1f_engine* e, int area) { return reinterpret_cast<double*>(e->h_res + (size_t)area * e->res_area_bytes); }
float* res_curve(const hw1f_engine* e, int area)
{
    return reinterpret_cast<float*>(e->h_res + (size_t)area * e->res_area_bytes + e->res_doubles * sizeof(double));
}

int make_tail(hw1f_engine* e, int n_runs, unsigned grid_x, uint64_t n_local, int nq, int ncur, const float* c0,
              const float* c1, float scale, double* d_moments, int out_stride, int n_ext_out, const Finish& fin, TailArgs* t)
{
    const unsigned n_groups = (grid_x + kTailGroup - 1) / kTailGroup;
    HW_REQUIRE(e, n_runs <= kTailCounters, "too many runs for the ticket counters");
    HW_CUDA(e, e->d_gpart.ensure((size_t)n_runs * n_groups * nq));
    memset(t, 0, sizeof(*t));
    t->counters = e->d_tail_cnt.p;
    t->gpart = e->d_gpart.p;
    t->moments = d_moments;
    t->host_mom = fin.host_mom;
    t->out_stride = out_stride;
    t->n_ext_out = n_ext_out;
    t->ncur = ncur;
    t->n_mat = e->p.n_mat;
    t->center0 = c0;
    t->center1 = c1;
    t->center_scale = scale;
    t->n_local = n_local;
    if (fin.exchange && e->comm_on) {
        HW_REQUIRE(e, n_runs == 1, "the peer exchange works on single-run launches");
        HW_REQUIRE(e, ncur * 2 * e->p.n_mat + n_ext_out <= kCommMaxCount, "moment vector too long for the peer mailboxes");
        if (*e->comm_epoch == 0xffffffffu) { e->err = "communicator exhausted (2^32 exchanges): create a new one"; return HW1F_ERR_COMM; }
        t->comm = e->comm;
        t->epoch = ++*e->comm_epoch;
    }
    t->epi = fin.epi ? 1 : 0;
    t->n_total = fin.n_total;
    t->inv_dT = 1.0f / e->spacing;   // host division, src/1:76
    t->dev_curve = fin.dev_curve;
    t->host_curve = fin.host_curve;
    t->plan = fin.plan;
    return HW1F_OK;
}

// the publication step alone (the *_finish entry points: the vector comes back from an external all-reduce)
int publish(hw1f_engine* e, int n_runs, int ncur, double* d_moments, int out_stride, int n_ext_out, const Finish& fin)
{
    if (!fin.host_mom && !(fin.exchange && e->comm_on) && !fin.epi) return HW1F_OK;
    TailArgs t;
    HW_TRY(make_tail(e, n_runs, 1, 0, 1, ncur, nullptr, nullptr, 0.f, d_moments, out_stride, n_ext_out, fin, &t));
    tail_publish_kernel<<<n_runs, 256, (size_t)e->p.n_mat * sizeof(float), e->stream>>>(t, model_dev(e), ncur * 2 * e->p.n_mat);
    return check_launch(e, "tail_publish_kernel");
}

// everything behind a simulation launch in ONE kernel (hw1f_tail.cuh), launched with programmatic stream serialisation:
// its blocks are resident, parked in griddepcontrol.wait, when the last simulation block retires
int launch_tail(hw1f_engine* e, const Launch& L, uint64_t n_local, int nq, int ncur, const float* c0, const float* c1,
                float scale, double* d_moments, int out_stride, int n_ext_out, const Finish& fin)
{
    TailArgs ta;
    HW_TRY(make_tail(e, L.n_runs, L.grid_x, n_local, nq, ncur, c0, c1, scale, d_moments, out_stride, n_ext_out, fin, &ta));
    const unsigned n_groups = (L.grid_x + kTailGroup - 1) / kTailGroup;
    const size_t smem = tail_smem_bytes(nq, e->p.n_mat);
    HW_REQUIRE(e, smem <= 48 * 1024, "moment vector too long for the tail kernel's shared memory");
    HW_CUDA(e, launch_k(tail_kernel, dim3(n_groups, L.n_runs), dim3(kTailThreads), smem, e->stream, true, ta, model_dev(e),
                        (const double*)e->d_partials.p, (int)L.grid_x, nq, ncur * 2 * e->p.n_mat));
    return check_launch(e, "tail_kernel");
}

// ---- Q1 launch: sums for NSCEN scenarios into d_moments[n_runs][nscen*2*n_mat] -----------------
// dump_steps > 0 (decomposed mode, two scenarios, dump_steps on a save point): the kernel also stores the noise
// state of every subsequence at that step into e->d_state (see fast_kernel DUMP)
int launch_curve(hw1f_engine* e, const Launch& L, const ScenDev* sc, int nscen, double* d_moments, int dump_steps = 0,
                 const Finish& fin = Finish(), int keep = 0)
{
    const int nm = e->p.n_mat, nq = nscen * 2 * nm;
    HW_CUDA(e, e->d_partials.ensure((size_t)L.n_runs * L.grid_x * nq));
    const dim3 grid(L.grid_x, L.n_runs);
    if (e->mode == HW1F_MODE_DECOMPOSED) {
        const int slot0 = drift_slot_of(e, sc[0]), slot1 = drift_slot_of(e, sc[nscen > 1 ? 1 : 0]);
        const FastScen c0 = fast_scen(e, sc[0].sig_st, slot0, 0), c1 = fast_scen(e, sc[nscen > 1 ? 1 : 0].sig_st, slot1, 0);
        const FastTangent tg{0.f, 0.f};
        const size_t smem = smem_fast(e, nscen, 0, 0);
        const ModelDev md = model_dev(e);
        if (e->stride & 1) {   // any save stride: the instantiations that may split a Box-Muller pair at a save point
            HW_REQUIRE(e, dump_steps == 0, "the one-pass recalibration needs an even save stride");
            if (nscen == 1) {
                HW_TRY(set_smem(e, (fast_kernel<1, 0, 0, 0, 0, 1>), smem));
                HW_CUDA(e, launch_k(fast_kernel<1, 0, 0, 0, 0, 1>, grid, kThreads, smem, e->stream, true, L.g, L.seeds, md, c0,
                                    c1, c0, c0, c0, tg, e->d_plans.p, 0, 0, 0.f, e->d_partials.p, (float2*)nullptr));
            } else {
                HW_TRY(set_smem(e, (fast_kernel<2, 0, 0, 0, 0, 1>), smem));
                HW_CUDA(e, launch_k(fast_kernel<2, 0, 0, 0, 0, 1>, grid, kThreads, smem, e->stream, true, L.g, L.seeds, md, c0,
                                    c1, c0, c0, c0, tg, e->d_plans.p, 0, 0, 0.f, e->d_partials.p, (float2*)nullptr));
            }
        } else if (nscen == 1) {
            HW_TRY(set_smem(e, fast_kernel<1, 0, 0>, smem));
            HW_CUDA(e, launch_k(fast_kernel<1, 0, 0>, grid, kThreads, smem, e->stream, true, L.g, L.seeds, md, c0, c1, c0, c0,
                                c0, tg, e->d_plans.p, 0, 0, 0.f, e->d_partials.p, (float2*)nullptr));
        } else if (dump_steps > 0) {
            HW_CUDA(e, e->d_state.ensure((size_t)L.n_runs * L.g.n_chunks * kChunk));
            HW_TRY(set_smem(e, (fast_kernel<2, 0, 0, 1>), smem));
            HW_CUDA(e, launch_k(fast_kernel<2, 0, 0, 1>, grid, kThreads, smem, e->stream, true, L.g, L.seeds, md, c0, c1, c0,
                                c0, c0, tg, e->d_plans.p, dump_steps, keep, 0.f, e->d_partials.p, e->d_state.p));
        } else {
            HW_TRY(set_smem(e, fast_kernel<2, 0, 0>, smem));
            HW_CUDA(e, launch_k(fast_kernel<2, 0, 0>, grid, kThreads, smem, e->stream, true, L.g, L.seeds, md, c0, c1, c0, c0,
                                c0, tg, e->d_plans.p, 0, 0, 0.f, e->d_partials.p, (float2*)nullptr));
        }
        HW_TRY(check_launch(e, "fast_kernel<curve>"));
        return launch_tail(e, L, L.g.n_paths, nq, nscen, c0.emI, c1.emI, 2.0f, d_moments, nq, 0, fin);
    }
    const size_t smem = smem_curve(e, nscen);
    if (e->stride & 1) {
        if (nscen == 1) {
            HW_TRY(set_smem(e, (bond_curve_kernel<1, 1>), smem));
            bond_curve_kernel<1, 1><<<grid, kThreads, smem, e->stream>>>(L.g, L.seeds, model_dev(e), sc[0], sc[0],
                                                                         e->d_partials.p);
        } else {
            HW_TRY(set_smem(e, (bond_curve_kernel<2, 1>), smem));
            bond_curve_kernel<2, 1><<<grid, kThreads, smem, e->stream>>>(L.g, L.seeds, model_dev(e), sc[0], sc[1],
                                                                         e->d_partials.p);
        }
    } else if (nscen == 1) {
        HW_TRY(set_smem(e, bond_curve_kernel<1>, smem));
        bond_curve_kernel<1><<<grid, kThreads, smem, e->stream>>>(L.g, L.seeds, model_dev(e), sc[0], sc[0],
                                                                  e->d_partials.p);
    } else {
        HW_TRY(set_smem(e, bond_curve_kernel<2>, smem));
        bond_curve_kernel<2><<<grid, kThreads, smem, e->stream>>>(L.g, L.seeds, model_dev(e), sc[0], sc[1],
                                                                  e->d_partials.p);
    }
    HW_TRY(check_launch(e, "bond_curve_kernel"));
    return launch_tail(e, L, L.g.n_paths, nq, nscen, sc[0].center, sc[nscen > 1 ? 1 : 0].center, 1.0f, d_moments, nq, 0, fin);
}

int launch_zbc(hw1f_engine* e, const Launch& L, const ScenDev* sc, int nscen, int n_steps_S1, float K,
               double* d_moments, const Finish& fin = Finish())
{
    const int nq = nscen * 5;
    HW_CUDA(e, e->d_partials.ensure((size_t)L.n_runs * L.grid_x * nq));
    const dim3 grid(L.grid_x, L.n_runs);
    if (e->mode == HW1F_MODE_DECOMPOSED) {
        const FastScen z0 = fast_scen(e, sc[0].sig_st, drift_slot_of(e, sc[0]), n_steps_S1);
        const FastScen z1 = fast_scen(e, sc[nscen > 1 ? 1 : 0].sig_st, drift_slot_of(e, sc[nscen > 1 ? 1 : 0]), n_steps_S1);
        const FastTangent tg{0.f, 0.f};
        const size_t smemf = smem_fast(e, 0, nscen, 0);
        const ModelDev md = model_dev(e);
        if (nscen == 1) {
            HW_TRY(set_smem(e, fast_kernel<0, 1, 0>, smemf));
            HW_CUDA(e, launch_k(fast_kernel<0, 1, 0>, grid, kThreads, smemf, e->stream, true, L.g, L.seeds, md, z0, z0, z0, z1,
                                z1, tg, e->d_plans.p, n_steps_S1, L.lead, K, e->d_partials.p, (float2*)nullptr));
        } else {
            HW_TRY(set_smem(e, fast_kernel<0, 2, 0>, smemf));
            HW_CUDA(e, launch_k(fast_kernel<0, 2, 0>, grid, kThreads, smemf, e->stream, true, L.g, L.seeds, md, z0, z0, z0, z1,
                                z1, tg, e->d_plans.p, n_steps_S1, L.lead, K, e->d_partials.p, (float2*)nullptr));
        }
        HW_TRY(check_launch(e, "fast_kernel<zbc>"));
    } else {
        const size_t smem = (size_t)kWinWords * 4 + (size_t)nscen * ((n_steps_S1 + 1) / 2 + 1) * sizeof(float4);
        if (nscen == 1) {
            HW_TRY(set_smem(e, zbc_kernel<1>, smem));
            zbc_kernel<1><<<grid, kThreads, smem, e->stream>>>(L.g, L.seeds, model_dev(e), sc[0], sc[0], e->d_plans.p,
                                                               n_steps_S1, L.lead, K, e->d_partials.p);
        } else {
            HW_TRY(set_smem(e, zbc_kernel<2>, smem));
            zbc_kernel<2><<<grid, kThreads, smem, e->stream>>>(L.g, L.seeds, model_dev(e), sc[0], sc[1], e->d_plans.p,
                                                               n_steps_S1, L.lead, K, e->d_partials.p);
        }
        HW_TRY(check_launch(e, "zbc_kernel"));
    }
    return launch_tail(e, L, L.g.n_paths, nq, 0, nullptr, nullptr, 0.f, d_moments, nq, nq, fin);
}

// the two ZBC scenarios evaluated on the noise state a preceding launch_curve(.., dump_steps = n_steps_S1) left in
// e->d_state: same moments as launch_zbc on the same normals, without simulating them again
int launch_zbc_from_state(hw1f_engine* e, const Launch& L, const ScenDev* sc, int n_steps_S1, float K, double* d_moments,
                          const Finish& fin = Finish())
{
    const int nq = 10;
    HW_CUDA(e, e->d_partials.ensure((size_t)L.n_runs * L.grid_x * nq));
    const FastScen z0 = fast_scen(e, sc[0].sig_st, drift_slot_of(e, sc[0]), n_steps_S1);
    const FastScen z1 = fast_scen(e, sc[1].sig_st, drift_slot_of(e, sc[1]), n_steps_S1);
    // behind the curve launch's tail kernel (which wrote the recalibrated curves' bond plans): ordinary stream order
    zbc_from_state_kernel<2><<<dim3(L.grid_x, L.n_runs), kThreads, 0, e->stream>>>(L.g, z0, z1, e->d_plans.p, K, e->d_state.p,
                                                                                  e->d_partials.p);
    HW_TRY(check_launch(e, "zbc_from_state_kernel"));
    return launch_tail(e, L, L.g.n_paths, nq, 0, nullptr, nullptr, 0.f, d_moments, nq, nq, fin);
}

int launch_pathwise(hw1f_engine* e, const Launch& L, const ScenDev& sc, int n_steps_S1, float K, double* d_moments,
                    const Finish& fin = Finish())
{
    HW_CUDA(e, e->d_partials.ensure((size_t)L.n_runs * L.grid_x * 3));
    if (e->mode == HW1F_MODE_DECOMPOSED) {
        const FastScen z0 = fast_scen(e, sc.sig_st, drift_slot_of(e, sc), n_steps_S1);
        const FastTangent tg = fast_tangent(e, n_steps_S1);
        const size_t smemf = smem_fast(e, 0, 0, 1);
        HW_TRY(set_smem(e, fast_kernel<0, 0, 1>, smemf));
        HW_CUDA(e, launch_k(fast_kernel<0, 0, 1>, dim3(L.grid_x, L.n_runs), kThreads, smemf, e->stream, true, L.g, L.seeds,
                            model_dev(e), z0, z0, z0, z0, z0, tg, e->d_plans.p, n_steps_S1, L.lead, K, e->d_partials.p,
                            (float2*)nullptr));
        HW_TRY(check_launch(e, "fast_kernel<pathwise>"));
        // the kernel keeps a third sum (for the fused form); the entry points emit sum v, sum v^2
        return launch_tail(e, L, L.g.n_paths, 3, 0, nullptr, nullptr, 0.f, d_moments, 2, 2, fin);
    }
    const size_t smem = (size_t)kWinWords * 4 + (size_t)(n_steps_S1 + 1) * sizeof(float4);
    HW_TRY(set_smem(e, pathwise_kernel, smem));
    pathwise_kernel<<<dim3(L.grid_x, L.n_runs), kThreads, smem, e->stream>>>(L.g, L.seeds, model_dev(e), sc,
                                                                            e->d_plans.p, n_steps_S1, L.lead, K,
                                                                            e->d_partials.p);
    HW_TRY(check_launch(e, "pathwise_kernel"));
    return launch_tail(e, L, L.g.n_paths, 2, 0, nullptr, nullptr, 0.f, d_moments, 2, 2, fin);
}

// a moment vector that went through a timed-out peer all-reduce is NaN-poisoned (hw1f_comm.cu)
int require_finite(hw1f_engine* e, const double* v, int n)
{
    for (int k = 0; k < n; ++k)
        if (!std::isfinite(v[k])) {
            e->err = "moment vector is not finite (a peer all-reduce timed out, see hw1f_comm_timeouts)";
            return HW1F_ERR_COMM;
        }
    return HW1F_OK;
}

// float32 host algebra of src/2:154-179 / :259-290 (+ double extras)
void zbc_algebra(const double mom[5], uint64_t n_paths_total, float P0S2, int32_t n_steps_S1, hw1f_zbc_result* r)
{
    memset(r, 0, sizeof(*r));
    for (int k = 0; k < 5; ++k) r->mom[k] = mom[k];
    // the reference divides by `int N_total` (src/2:154): the same value as a float for every count an int
    // can hold; beyond 2^31 - 1 (multi-GPU scaling run) the float algebra simply continues with (float)N
    const float N_total = (float)(2 * n_paths_total);
    r->n_total = 2 * n_paths_total;
    r->n_steps_S1 = n_steps_S1;
    const float h_ZBC = (float)mom[0], h_control = (float)mom[1], h_ZBC_sq = (float)mom[2],
                h_control_sq = (float)mom[3], h_cross = (float)mom[4];
    const float mean_ZBC = h_ZBC / N_total;
    const float mean_control = h_control / N_total;
    const float E_Y2 = h_control_sq / N_total;
    const float E_Y_sq = mean_control * mean_control;
    const float var_control = E_Y2 - E_Y_sq;
    const float E_XY = h_cross / N_total;
    const float E_X_E_Y = mean_ZBC * mean_control;
    const float cov = E_XY - E_X_E_Y;
    const float beta = cov / var_control;
    const float control_adjustment = beta * (mean_control - P0S2);
    const float adjusted = mean_ZBC - control_adjustment;
    const float corr_single = cov / (sqrtf(var_control) * sqrtf(E_Y2 - E_Y_sq));
    const float E_X2 = h_ZBC_sq / N_total;
    const float var_ZBC = E_X2 - mean_ZBC * mean_ZBC;
    const float corr = cov / sqrtf(var_ZBC * var_control);
    r->mean_X = mean_ZBC; r->mean_Y = mean_control; r->var_X = var_ZBC; r->var_Y = var_control;
    r->cov = cov; r->beta = beta; r->control_adjustment = control_adjustment;
    r->price_raw = mean_ZBC; r->price_cv = adjusted; r->corr_single = corr_single; r->corr = corr;
    // double-precision companions.  The per-thread samples are antithetic pair sums, so the
    // i.i.d. unit is the pair: x = X/2, y = Y/2 with n = n_paths_total samples.
    const double n = (double)n_paths_total;
    const double mx = mom[0] / (2.0 * n), my = mom[1] / (2.0 * n);
    const double vyy = mom[3] / (2.0 * n) - my * my, cxy = mom[4] / (2.0 * n) - mx * my;
    const double b = (vyy > 0) ? cxy / vyy : 0.0;
    r->beta_f64 = b;
    r->price_cv_f64 = mx - b * (my - (double)P0S2);
    // standard errors: per-path second moments are an upper bound for the pair-mean variance
    const double vxx = mom[2] / (2.0 * n) - mx * mx;
    const double var_cv = vxx - 2.0 * b * cxy + b * b * vyy;
    r->se_raw = (vxx > 0) ? sqrt(vxx / (2.0 * n)) : 0.0;
    r->se_cv = (var_cv > 0) ? sqrt(var_cv / (2.0 * n)) : 0.0;
    r->ci95_lo = r->price_cv_f64 - 1.959963984540054 * r->se_cv;
    r->ci95_hi = r->price_cv_f64 + 1.959963984540054 * r->se_cv;
    // beta*, rho and their standard errors from the same five moments: regression slope and Fisher's formula with one
    // degree of freedom per antithetic pair
    const double rho = (vxx > 0 && vyy > 0) ? cxy / sqrt(vxx * vyy) : 0.0;
    r->corr_f64 = rho;
    r->beta_se = (vyy > 0 && n > 2) ? sqrt((1.0 - rho * rho) * vxx / (vyy * (n - 2.0))) : 0.0;
    r->corr_se = (n > 3) ? (1.0 - rho * rho) / sqrt(n - 3.0) : 0.0;
}

// loads every simulation kernel and opts it in to the full shared-memory carve-out (once per engine)
int init_kernels(hw1f_engine* e)
{
    const size_t b = e->smem_optin;
    HW_CUDA(e, opt_in(bond_curve_kernel<1>, b));
    HW_CUDA(e, opt_in(bond_curve_kernel<2>, b));
    HW_CUDA(e, opt_in(zbc_kernel<1>, b));
    HW_CUDA(e, opt_in(zbc_kernel<2>, b));
    HW_CUDA(e, opt_in(pathwise_kernel, b));
    HW_CUDA(e, opt_in(fused_kernel<false>, b));
    HW_CUDA(e, opt_in(fused_kernel<true>, b));
    HW_CUDA(e, opt_in(fast_kernel<1, 0, 0>, b));
    HW_CUDA(e, opt_in(fast_kernel<2, 0, 0>, b));
    HW_CUDA(e, opt_in((fast_kernel<2, 0, 0, 1>), b));
    HW_CUDA(e, opt_in(fast_kernel<0, 1, 0>, b));
    HW_CUDA(e, opt_in(fast_kernel<0, 2, 0>, b));
    HW_CUDA(e, opt_in(fast_kernel<0, 0, 1>, b));
    HW_CUDA(e, opt_in(fast_kernel<1, 1, 2>, b));
    HW_CUDA(e, opt_in(fast_kernel<1, 3, 2>, b));
    HW_CUDA(e, opt_in((fast_kernel<2, 3, 1, 1, 1>), b));
    HW_CUDA(e, opt_in((fast_kernel<1, 0, 0, 0, 0, 1>), b));
    HW_CUDA(e, opt_in((fast_kernel<2, 0, 0, 0, 0, 1>), b));
    HW_CUDA(e, opt_in((bond_curve_kernel<1, 1>), b));
    HW_CUDA(e, opt_in((bond_curve_kernel<2, 1>), b));
    HW_CUDA(e, opt_in(zbc_sum_kernel<0>, b));
    HW_CUDA(e, opt_in(zbc_sum_kernel<1>, b));
    HW_CUDA(e, opt_in(zbc_sum_kernel<2>, b));
    HW_CUDA(e, opt_in(zbc_sum_kernel<3>, b));
    HW_CUDA(e, opt_in(cap_kernel<0>, b));
    HW_CUDA(e, opt_in(cap_kernel<1>, b));
    HW_CUDA(e, opt_in(swaption_kernel<0>, b));
    HW_CUDA(e, opt_in(swaption_kernel<1>, b));
    // the small kernels have no dynamic shared memory; querying them loads their code now instead
    // of inside the first timed call
    cudaFuncAttributes attr;
    HW_CUDA(e, cudaFuncGetAttributes(&attr, prep_lo_kernel));
    HW_CUDA(e, cudaFuncGetAttributes(&attr, build_hi_kernel));
    HW_CUDA(e, cudaFuncGetAttributes(&attr, plan_job_kernel));
    HW_CUDA(e, cudaFuncGetAttributes(&attr, tail_publish_kernel));
    HW_CUDA(e, cudaFuncGetAttributes(&attr, tail_kernel));
    HW_CUDA(e, cudaFuncGetAttributes(&attr, reduce_partials_kernel<double>));
    HW_CUDA(e, cudaFuncGetAttributes(&attr, zbc_from_state_kernel<2>));
    HW_CUDA(e, cudaFuncGetAttributes(&attr, curve_epilogue_kernel));
    HW_CUDA(e, cudaFuncGetAttributes(&attr, theta_kernel));
    HW_CUDA(e, cudaFuncGetAttributes(&attr, sample_paths_kernel));
    HW_CUDA(e, cudaFuncGetAttributes(&attr, steps_probe_kernel));
    // ticket counters of the kernel tails (self-resetting: zeroed once), bond plans
    HW_CUDA(e, e->d_tail_cnt.ensure(kTailCounters));
    HW_CUDA(e, cudaMemsetAsync(e->d_tail_cnt.p, 0, kTailCounters * sizeof(unsigned), e->stream));
    HW_CUDA(e, e->d_plans.ensure(4));
    return ensure_tables(e);
}

// seed-independent tables for a handle's path range (built once, cached): keeps one-off work out
// of the event-timed region of the public calls
int warm_geometry(hw1f_engine* e, const hw1f_rng* rng)
{
    HW_TRY(ensure_tables(e));
    const uint32_t L_log2 = pick_L_log2(rng->n_paths);
    const uint64_t last_path = rng->first_path + rng->n_paths - 1;
    HW_REQUIRE(e, (last_path >> L_log2) < (1ull << 32), "path index too large for the jump tables (>= 2^41)");
    HW_TRY(ensure_windows(e, L_log2, (uint32_t)(rng->first_path >> L_log2), (uint32_t)(last_path >> L_log2)));
    // scratch every single-seed launch over this range will need (cudaMalloc is not free either)
    HW_CUDA(e, e->d_U.ensure((size_t)5 << L_log2));
    const unsigned long long n_chunks = (last_path >> kChunkLog2) - (rng->first_path >> kChunkLog2) + 1;
    const unsigned long long cap = (unsigned long long)e->sm_count * 32ull;
    const size_t grid = (size_t)(n_chunks < cap ? n_chunks : cap);
    if (e->has_model) HW_CUDA(e, e->d_partials.ensure(grid * (4 * (size_t)e->p.n_mat + 32)));
    return HW1F_OK;
}

}  // namespace

// =================================================================================================
// C ABI
// =================================================================================================
extern "C" {

int hw1f_abi_version(void) { return HW1F_ABI_VERSION; }

const char* hw1f_status_string(int s)
{
    switch (s) {
        case HW1F_OK: return "ok";
        case HW1F_ERR_INVALID: return "invalid argument";
        case HW1F_ERR_CUDA: return "CUDA error";
        case HW1F_ERR_NO_DEVICE: return "no CUDA device";
        case HW1F_ERR_UNSUPPORTED: return "unsupported configuration";
        case HW1F_ERR_NO_MODEL: return "model not set";
        case HW1F_ERR_COMM: return "moment vector not finite (peer all-reduce timed out)";
        default: return "unknown status";
    }
}

const char* hw1f_last_error(const hw1f_engine* e) { return e ? e->err.c_str() : "null engine"; }

int hw1f_engine_create(int device, hw1f_engine** out)
{
    if (!out) return HW1F_ERR_INVALID;
    *out = nullptr;
    int count = 0;
    if (cudaGetDeviceCount(&count) != cudaSuccess || count <= 0) { cudaGetLastError(); return HW1F_ERR_NO_DEVICE; }
    if (device < 0) {   // select_gpu(), common.cuh:122-141
        size_t best_free = 0;
        device = 0;
        for (int i = 0; i < count; ++i) {
            size_t fr = 0, tot = 0;
            if (cudaSetDevice(i) == cudaSuccess && cudaMemGetInfo(&fr, &tot) == cudaSuccess && fr > best_free) {
                best_free = fr;
                device = i;
            }
        }
    }
    if (device >= count) return HW1F_ERR_NO_DEVICE;
    hw1f_engine* e = new (std::nothrow) hw1f_engine();
    if (!e) return HW1F_ERR_INVALID;
    e->device = device;
    cudaDeviceProp prop;
    if (cudaSetDevice(device) != cudaSuccess || cudaGetDeviceProperties(&prop, device) != cudaSuccess) {
        delete e;
        return HW1F_ERR_CUDA;
    }
    if (prop.major < 10) {   // sm_100a binary only: fail loudly instead of a confusing launch error
        delete e;
        return HW1F_ERR_UNSUPPORTED;
    }
    e->sm_count = prop.multiProcessorCount;
    e->smem_optin = prop.sharedMemPerBlockOptin;
    if (cudaStreamCreateWithFlags(&e->own_stream, cudaStreamNonBlocking) != cudaSuccess ||
        cudaEventCreate(&e->ev0) != cudaSuccess || cudaEventCreate(&e->ev1) != cudaSuccess ||
        cudaEventCreate(&e->ev2) != cudaSuccess || cudaEventCreate(&e->ev3) != cudaSuccess ||
        cudaEventCreateWithFlags(&e->ev_stage, cudaEventDisableTiming) != cudaSuccess ||
        cudaEventCreateWithFlags(&e->ev_fd, cudaEventDisableTiming) != cudaSuccess) {
        delete e;
        return HW1F_ERR_CUDA;
    }
    for (auto& ev : e->ev_slot)
        if (cudaEventCreateWithFlags(&ev, cudaEventDisableTiming) != cudaSuccess) {
            hw1f_engine_destroy(e);
            return HW1F_ERR_CUDA;
        }
    e->stream = e->own_stream;
    if (const char* q = std::getenv("HW1F_Q3_ONE_LAUNCH")) e->seq_one_launch = q[0] != '0';
    if (init_kernels(e) != HW1F_OK) {
        std::fprintf(stderr, "hw1f_engine_create: %s\n", e->err.c_str());
        hw1f_engine_destroy(e);
        return HW1F_ERR_CUDA;
    }
    *out = e;
    return HW1F_OK;
}

int hw1f_engine_destroy(hw1f_engine* e)
{
    if (!e) return HW1F_OK;
    for (auto& t : e->twin) {
        if (t) hw1f_engine_destroy(t);
        t = nullptr;
    }
    cudaSetDevice(e->device);
    cudaStreamSynchronize(e->stream);
    e->d_Jpow2.release(); e->d_Jnib.release(); e->d_W.release(); e->d_U.release();
    for (auto& d : e->d_drift) d.release();
    e->d_mkt.release(); e->d_center.release(); e->d_plans.release();
    for (auto& d : e->d_emI) d.release(); e->d_partials.release(); e->d_moments.release(); e->d_state.release();
    e->d_out.release(); e->d_int.release(); e->d_cap.release();
    e->d_model.release();
    e->d_fd.release();
    e->d_tail_cnt.release(); e->d_gpart.release();
    if (e->h_res) cudaFreeHost(e->h_res);
    if (e->h_model) cudaFreeHost(e->h_model);
    if (e->h_fd) cudaFreeHost(e->h_fd);
    if (e->ev_fd) cudaEventDestroy(e->ev_fd);
    if (e->h_stage) cudaFreeHost(e->h_stage);
    if (e->ev0) cudaEventDestroy(e->ev0);
    if (e->ev1) cudaEventDestroy(e->ev1);
    if (e->ev2) cudaEventDestroy(e->ev2);
    if (e->ev3) cudaEventDestroy(e->ev3);
    if (e->ev_stage) cudaEventDestroy(e->ev_stage);
    for (auto ev : e->ev_slot) if (ev) cudaEventDestroy(ev);
    if (e->own_stream) cudaStreamDestroy(e->own_stream);
    delete e;
    return HW1F_OK;
}

int hw1f_engine_set_stream(hw1f_engine* e, void* s)
{
    if (!e) return HW1F_ERR_INVALID;
    HW_CUDA(e, cudaSetDevice(e->device));
    HW_CUDA(e, cudaStreamSynchronize(e->stream));
    e->stream = s ? (cudaStream_t)s : e->own_stream;
    return HW1F_OK;
}

int hw1f_engine_set_mode(hw1f_engine* e, int mode)
{
    if (!e) return HW1F_ERR_INVALID;
    HW_REQUIRE(e, mode == HW1F_MODE_REFERENCE_ORDER || mode == HW1F_MODE_DECOMPOSED, "unknown mode");
    e->mode = mode;
    return HW1F_OK;
}

int hw1f_engine_get_mode(const hw1f_engine* e, int* mode)
{
    if (!e || !mode) return HW1F_ERR_INVALID;
    *mode = e->mode;
    return HW1F_OK;
}

int hw1f_engine_device(const hw1f_engine* e, int* d)
{
    if (!e || !d) return HW1F_ERR_INVALID;
    *d = e->device;
    return HW1F_OK;
}

int hw1f_engine_synchronize(hw1f_engine* e)
{
    if (!e) return HW1F_ERR_INVALID;
    HW_CUDA(e, cudaSetDevice(e->device));
    HW_CUDA(e, cudaStreamSynchronize(e->stream));
    for (auto t : e->twin) if (t) HW_CUDA(e, cudaStreamSynchronize(t->stream));
    return HW1F_OK;
}

int hw1f_default_params(hw1f_params* p)
{
    if (!p) return HW1F_ERR_INVALID;
    p->a = 1.0f; p->sigma = 0.1f; p->r0 = 0.012f;            // common.cuh:37-39
    p->T_final = 10.0f; p->n_steps = 1000; p->n_mat = 101;   // common.cuh:16-22
    p->theta_a0 = 0.012f; p->theta_b0 = 0.0014f;             // common.cuh:229
    p->theta_a1 = 0.019f; p->theta_b1 = 0.001f;
    p->theta_break = 5.0f;
    p->fd_theta_a1 = 0.014f;                                 // src/3:387
    return HW1F_OK;
}

int hw1f_set_model(hw1f_engine* e, const hw1f_params* p)
{
    if (!e || !p) return HW1F_ERR_INVALID;
    HW_REQUIRE(e, p->n_mat >= 3 && p->n_mat <= 1024, "n_mat must be in [3,1024]");
    HW_REQUIRE(e, p->n_steps >= 2 && p->n_steps <= 8192, "n_steps must be in [2,8192]");
    HW_REQUIRE(e, p->n_steps % (p->n_mat - 1) == 0, "N_STEPS must be evenly divisible by (N_MAT - 1)");  // common.cuh:25-27
    HW_REQUIRE(e, p->a > 0.0f && p->sigma > 0.0f && p->T_final > 0.0f, "a, sigma, T_final must be positive");
    HW_CUDA(e, cudaSetDevice(e->device));
    const int n = p->n_steps, nm = p->n_mat;
    // arena layout (256-byte aligned pieces): drift2[0], drift2[1], centre[nm], emI[nm]
    auto align = [](size_t x) { return (x + 255) & ~(size_t)255; };
    const size_t off_d0 = 0, off_d1 = align((size_t)(n + 2) * sizeof(float2));
    const size_t off_c = off_d1 + align((size_t)(n + 2) * sizeof(float2));
    const size_t off_e = off_c + align((size_t)nm * sizeof(float));
    const size_t total = off_e + align((size_t)nm * sizeof(float));
    e->model_off_emI = off_e;
    const bool same = e->model_cached && memcmp(&e->cached_p, p, sizeof(*p)) == 0 && total == e->model_bytes;
    if (!same) {
        // an upload enqueued by an earlier call may still read the pinned mirror
        HW_CUDA(e, cudaStreamSynchronize(e->stream));
        if (total != e->model_bytes) {
            HW_CUDA(e, cudaStreamSynchronize(e->stream));
            e->d_drift[0].release(); e->d_drift[1].release(); e->d_center.release(); e->d_emI[0].release();
            e->d_model.release();
            if (e->h_model) cudaFreeHost(e->h_model);
            e->h_model = nullptr;
            e->model_bytes = 0;
            HW_CUDA(e, e->d_model.ensure(total));
            HW_CUDA(e, cudaMallocHost((void**)&e->h_model, total));
            e->model_bytes = total;
            e->d_drift[0].set_view(reinterpret_cast<float2*>(e->d_model.p + off_d0), n + 2);
            e->d_drift[1].set_view(reinterpret_cast<float2*>(e->d_model.p + off_d1), n + 2);
            e->d_center.set_view(reinterpret_cast<float*>(e->d_model.p + off_c), nm);
            e->d_emI[0].set_view(reinterpret_cast<float*>(e->d_model.p + off_e), nm);
        }
        e->p = *p;
        e->dt = p->T_final / p->n_steps;                  // H_DT, common.cuh:33
        e->spacing = p->T_final / (p->n_mat - 1);         // H_MAT_SPACING, common.cuh:34
        e->exp_adt = expf(-p->a * e->dt);                 // common.cuh:93
        e->sig_st = host_sig_st(*p, p->sigma);            // common.cuh:94
        e->stride = p->n_steps / (p->n_mat - 1);          // SAVE_STRIDE, common.cuh:29
        e->h_drift.assign(n, 0.f);
        e->h_sdrift.assign(n, 0.f);
        host_drift_tables(*p, p->sigma, e->h_drift.data(), e->h_sdrift.data());
        memset(e->h_model, 0, total);
        float2* d0 = reinterpret_cast<float2*>(e->h_model + off_d0);
        float2* d1 = reinterpret_cast<float2*>(e->h_model + off_d1);
        for (int i = 0; i < n; ++i) {
            d0[i] = make_float2(e->h_drift[i], e->h_drift[i]);
            d1[i] = make_float2(e->h_sdrift[i], e->h_sdrift[i]);
        }
        float* cen = reinterpret_cast<float*>(e->h_model + off_c);
        float* emI = reinterpret_cast<float*>(e->h_model + off_e);
        build_det_tables(e, 0, e->h_drift.data(), emI);
        build_det_tables(e, 1, e->h_sdrift.data(), nullptr);
        // centring constants of the reference-order curve kernel: c_m = 2 exp(-I_m) along the noise-free path
        for (int k = 0; k < nm; ++k) cen[k] = 2.0f * emI[k];
        e->cached_p = *p;
        e->model_cached = true;
        e->fd_cached = false;      // the bumped-sigma tables and the step probe depend on the model
        e->steps_cached = false;
    }
    {   // result areas: the longest moment vector (two curve scenarios + extras) and P, f, P_se of two curves
        const size_t nd = (4 * (size_t)nm + 64 > 512) ? 4 * (size_t)nm + 64 : 512, nf = 6 * (size_t)nm;
        const size_t bytes = align(nd * sizeof(double) + nf * sizeof(float));
        if (bytes != e->res_area_bytes) {
            for (bool busy : e->slot_busy)
                HW_REQUIRE(e, !busy, "hw1f_set_model: n_mat changes the result areas while submissions are in flight (collect them first)");
            HW_CUDA(e, cudaStreamSynchronize(e->stream));
            if (e->h_res) cudaFreeHost(e->h_res);
            e->h_res = nullptr;
            e->res_area_bytes = 0;
            HW_CUDA(e, cudaHostAlloc((void**)&e->h_res, kResAreas * bytes, cudaHostAllocMapped));
            e->res_area_bytes = bytes;
            e->res_doubles = nd;
        }
    }
    e->has_model = true;
    ++e->model_gen;
    // compute_constants(): ONE host->device copy of the model tables (every call, like the reference's
    // cudaMemcpyToSymbol sequence; only the host-side table building is cached)
    HW_CUDA(e, cudaMemcpyAsync(e->d_model.p, e->h_model, total, cudaMemcpyHostToDevice, e->stream));
    return HW1F_OK;
}

int hw1f_get_model(const hw1f_engine* e, hw1f_params* out)
{
    if (!e || !out || !e->has_model) return HW1F_ERR_INVALID;
    *out = e->p;
    return HW1F_OK;
}

int hw1f_get_constants(const hw1f_engine* e, hw1f_constants* c)
{
    if (!e || !c || !e->has_model) return HW1F_ERR_INVALID;
    c->dt = e->dt; c->mat_spacing = e->spacing; c->exp_adt = e->exp_adt; c->sig_st = e->sig_st;
    c->save_stride = e->stride;
    return HW1F_OK;
}

int hw1f_get_drift_table(const hw1f_engine* e, int which, float sigma, float* out)
{
    if (!e || !out || !e->has_model) return HW1F_ERR_INVALID;
    if (which == 0) host_drift_tables(e->p, sigma, out, nullptr);
    else if (which == 1) host_drift_tables(e->p, sigma, nullptr, out);
    else if (which == 2) host_shifted_drift_table(e->p, sigma, e->p.sigma, out);
    else return HW1F_ERR_INVALID;
    return HW1F_OK;
}

int hw1f_steps_to(hw1f_engine* e, float S1, int32_t* n)
{
    HW_TRY(require_model(e));
    if (!n) return HW1F_ERR_INVALID;
    if (e->steps_cached && e->steps_S1 == S1 && e->steps_dt == e->dt) { *n = e->steps_n; return HW1F_OK; }
    HW_CUDA(e, cudaSetDevice(e->device));
    HW_CUDA(e, e->d_int.ensure(4));
    steps_probe_kernel<<<1, 1, 0, e->stream>>>(S1, e->dt, e->d_int.p);
    HW_TRY(check_launch(e, "steps_probe_kernel"));
    int v = 0;
    HW_TRY(download(e, &v, e->d_int.p, sizeof(int)));
    *n = v;
    e->steps_cached = true;    // the device expression is a pure function of (S1, dt)
    e->steps_S1 = S1;
    e->steps_dt = e->dt;
    e->steps_n = v;
    return HW1F_OK;
}

// ---- RNG handle ------------------------------------------------------------------------------
int hw1f_rng_create(uint64_t seed, uint64_t first_path, uint64_t n_paths, hw1f_rng** out)
{
    if (!out || n_paths == 0) return HW1F_ERR_INVALID;
    hw1f_rng* r = new (std::nothrow) hw1f_rng{seed, first_path, n_paths, 0};
    if (!r) return HW1F_ERR_INVALID;
    *out = r;
    return HW1F_OK;
}
int hw1f_rng_clone(const hw1f_rng* src, hw1f_rng** out)
{
    if (!src || !out) return HW1F_ERR_INVALID;
    *out = new (std::nothrow) hw1f_rng(*src);
    return *out ? HW1F_OK : HW1F_ERR_INVALID;
}
int hw1f_rng_destroy(hw1f_rng* r) { delete r; return HW1F_OK; }
int hw1f_rng_tell(const hw1f_rng* r, uint64_t* off)
{
    if (!r || !off) return HW1F_ERR_INVALID;
    *off = r->offset;
    return HW1F_OK;
}
int hw1f_rng_seek(hw1f_rng* r, uint64_t off)
{
    if (!r) return HW1F_ERR_INVALID;
    r->offset = off;
    return HW1F_OK;
}
int hw1f_rng_info(const hw1f_rng* r, uint64_t* seed, uint64_t* first, uint64_t* n)
{
    if (!r) return HW1F_ERR_INVALID;
    if (seed) *seed = r->seed;
    if (first) *first = r->first_path;
    if (n) *n = r->n_paths;
    return HW1F_OK;
}

int hw1f_rng_prepare(hw1f_engine* e, const hw1f_rng* rng)
{
    if (!e || !rng) return HW1F_ERR_INVALID;
    HW_CUDA(e, cudaSetDevice(e->device));
    return warm_geometry(e, rng);
}

// ---- Q1 ----------------------------------------------------------------------------------------
// stream-ordered wait + the host's view of a result area
static int wait_results(hw1f_engine* e)
{
    HW_CUDA(e, cudaStreamSynchronize(e->stream));
    return HW1F_OK;
}

static int curve_run(hw1f_engine* e, hw1f_rng* rng, double* d_moments, const Finish& fin)
{
    if (rng->offset & 1) {
        e->err = "bond curve needs an even normal offset (it starts on a Box-Muller pair boundary)";
        return HW1F_ERR_UNSUPPORTED;
    }
    Launch L;
    HW_TRY(prepare_launch(e, &rng->seed, 1, rng->first_path, rng->n_paths, rng->offset, &L));
    const ScenDev sc = scen_dev(e, e->p.sigma, e->sig_st, 0);
    HW_TRY(launch_curve(e, L, &sc, 1, d_moments, 0, fin));
    rng->offset += (uint64_t)e->p.n_steps;
    e->ci_valid = true;
    e->ci_geom = L.g;
    e->ci_blocks = L.grid_x;
    return HW1F_OK;
}

static int read_curve(hw1f_engine* e, int area, int scen, float* P, float* f, float* P_se)
{
    const int n = e->p.n_mat;
    const float* h = res_curve(e, area) + (size_t)scen * 3 * n;
    for (int k = 0; k < n; ++k)
        if (!std::isfinite(h[k])) {
            e->err = "moment vector is not finite (a peer all-reduce timed out, see hw1f_comm_timeouts)";
            return HW1F_ERR_COMM;
        }
    memcpy(P, h, n * sizeof(float));
    memcpy(f, h + n, n * sizeof(float));
    if (P_se) memcpy(P_se, h + 2 * n, n * sizeof(float));
    return HW1F_OK;
}

int hw1f_bond_curve_moments(hw1f_engine* e, hw1f_rng* rng, double* d_moments)
{
    HW_TRY(require_model(e));
    if (!rng || !d_moments) return HW1F_ERR_INVALID;
    HW_CUDA(e, cudaSetDevice(e->device));
    Finish fin;
    fin.exchange = true;   // with peers attached (hw1f_comm_attach) the last block all-reduces the vector itself
    return curve_run(e, rng, d_moments, fin);
}

int hw1f_bond_curve_finish(hw1f_engine* e, const double* d_moments, uint64_t n_paths_total, float* P, float* f,
                           float* P_se)
{
    HW_TRY(require_model(e));
    if (!d_moments || !P || !f) return HW1F_ERR_INVALID;
    HW_REQUIRE(e, n_paths_total >= 1 && n_paths_total < (1ull << 40), "n_paths_total outside [1, 2^40)");
    HW_CUDA(e, cudaSetDevice(e->device));
    Finish fin;
    fin.epi = true;
    fin.n_total = n_paths_total;
    fin.host_curve = res_curve(e, 0);
    HW_TRY(publish(e, 1, 1, const_cast<double*>(d_moments), 2 * e->p.n_mat, 0, fin));
    HW_TRY(wait_results(e));
    return read_curve(e, 0, 0, P, f, P_se);
}

int hw1f_bond_curve(hw1f_engine* e, hw1f_rng* rng, float* P, float* f, float* P_se, float* sim_ms)
{
    HW_TRY(require_model(e));
    if (!rng || !P || !f) return HW1F_ERR_INVALID;
    HW_CUDA(e, cudaSetDevice(e->device));
    HW_CUDA(e, e->d_moments.ensure(4 * (size_t)e->p.n_mat * kMaxRuns));
    HW_TRY(warm_geometry(e, rng));
    // one jump-table launch and ONE simulation launch whose last block reduces, finalises and stores P, f, P_se into
    // mapped pinned host memory; the host waits for the stream
    Finish fin;
    fin.epi = true;
    fin.n_total = rng->n_paths;
    fin.host_curve = res_curve(e, 0);
    if (sim_ms) HW_CUDA(e, cudaEventRecord(e->ev0, e->stream));
    HW_TRY(curve_run(e, rng, e->d_moments.p, fin));
    if (sim_ms) HW_CUDA(e, cudaEventRecord(e->ev1, e->stream));
    HW_TRY(wait_results(e));
    HW_TRY(read_curve(e, 0, 0, P, f, P_se));
    if (sim_ms) HW_CUDA(e, cudaEventElapsedTime(sim_ms, e->ev0, e->ev1));
    return HW1F_OK;
}

// hw1f_bond_curve in two halves: everything is enqueued by submit, collect waits for the slot's event only.  Slot 0
// runs on this engine's stream, the other slots on their twins': lanes whose kernels the GPU overlaps.
static int lane_of(hw1f_engine* e, int32_t slot, hw1f_engine** lane)
{
    *lane = e;
    if (slot == 0) return HW1F_OK;
    if (!e->twin[slot]) {
        const int st = hw1f_engine_create(e->device, &e->twin[slot]);
        if (st != HW1F_OK) { e->err = "could not create a submission lane"; return st; }
        e->twin_gen[slot] = 0;
    }
    hw1f_engine* t = e->twin[slot];
    t->mode = e->mode;
    if (e->twin_gen[slot] != e->model_gen) {   // every hw1f_set_model of the caller reaches the lane that runs the next call
        const int st = hw1f_set_model(t, &e->p);
        if (st != HW1F_OK) { e->err = t->err; return st; }
        e->twin_gen[slot] = e->model_gen;
    }
    *lane = t;
    return HW1F_OK;
}

int hw1f_bond_curve_submit(hw1f_engine* e, hw1f_rng* rng, int32_t slot)
{
    HW_TRY(require_model(e));
    if (!rng) return HW1F_ERR_INVALID;
    HW_REQUIRE(e, slot >= 0 && slot < kAsyncSlots, "slot outside [0, HW1F_ASYNC_SLOTS)");
    HW_REQUIRE(e, !e->slot_busy[slot], "result slot still in flight: collect it first");
    HW_CUDA(e, cudaSetDevice(e->device));
    hw1f_engine* t = nullptr;
    HW_TRY(lane_of(e, slot, &t));
    int st = HW1F_OK;
    auto run = [&]() -> int {
        HW_CUDA(t, t->d_moments.ensure(4 * (size_t)t->p.n_mat * kMaxRuns));
        HW_TRY(warm_geometry(t, rng));
        Finish fin;
        fin.epi = true;
        fin.n_total = rng->n_paths;
        fin.host_curve = res_curve(t, kSyncAreas + slot);
        HW_TRY(curve_run(t, rng, t->d_moments.p, fin));
        HW_CUDA(t, cudaEventRecord(t->ev_slot[slot], t->stream));
        return HW1F_OK;
    };
    st = run();
    if (st != HW1F_OK) {
        if (t != e) e->err = t->err;
        return st;
    }
    e->slot_busy[slot] = true;
    return HW1F_OK;
}

int hw1f_bond_curve_collect(hw1f_engine* e, int32_t slot, float* P, float* f, float* P_se)
{
    if (!e || !P || !f) return HW1F_ERR_INVALID;
    HW_REQUIRE(e, slot >= 0 && slot < kAsyncSlots, "slot outside [0, HW1F_ASYNC_SLOTS)");
    HW_REQUIRE(e, e->slot_busy[slot], "nothing was submitted to this result slot");
    HW_CUDA(e, cudaSetDevice(e->device));
    hw1f_engine* t = slot ? e->twin[slot] : e;
    HW_CUDA(e, cudaEventSynchronize(t->ev_slot[slot]));
    e->slot_busy[slot] = false;
    const int st = read_curve(t, kSyncAreas + slot, 0, P, f, P_se);
    if (st != HW1F_OK && t != e) e->err = t->err;
    return st;
}

// Standard errors of f(0,T) and theta(T) (and, as a cross-check, of P) by batch means over the simulation blocks of
// the last bond-curve launch + the delta method through compute_average_and_forward (market_data.cuh:101-127) and
// recover_theta (src/2:14-35): f and theta are linear in ln P of up to five neighbouring maturities.
int hw1f_bond_curve_ci(hw1f_engine* e, float* f_se, float* theta_se, float* P_se_batch)
{
    HW_TRY(require_model(e));
    HW_CUDA(e, cudaSetDevice(e->device));
    if (!e->ci_valid) {
        e->err = "hw1f_bond_curve_ci needs a preceding bond-curve launch on this engine (its block partials)";
        return HW1F_ERR_INVALID;
    }
    const int nm = e->p.n_mat;
    const unsigned B = e->ci_blocks;
    if (B < 8) {
        e->err = "batch-means confidence intervals need at least 8 simulation blocks (8192 subsequences)";
        return HW1F_ERR_UNSUPPORTED;
    }
    DevBuf<double> buf;
    HW_CUDA(e, buf.ensure((size_t)(kCiLags + 1) * nm));
    curve_batch_cov_kernel<<<nm, 256, 0, e->stream>>>(e->d_partials.p, (int)B, 2 * nm, nm, e->ci_geom, buf.p);
    int st = check_launch(e, "curve_batch_cov_kernel");
    std::vector<double> h((size_t)(kCiLags + 1) * nm);
    if (st == HW1F_OK) st = download(e, h.data(), buf.p, h.size() * sizeof(double));
    buf.release();
    HW_TRY(st);
    const double n = (double)e->ci_geom.n_paths, bias = (double)B / (double)(B - 1);
    const float* emI = reinterpret_cast<const float*>(e->h_model + e->model_off_emI);
    // P_m = (sum_b S_b[m] + n c_m) / (2n), c_m = 2 exp(-Im) (both arithmetic modes centre on it)
    std::vector<double> P(nm);
    for (int m = 0; m < nm; ++m) P[m] = (m == 0) ? 1.0 : (h[(size_t)kCiLags * nm + m] + n * 2.0 * (double)emI[m]) / (2.0 * n);
    // covariance of ln P_i, ln P_j for |i - j| < kCiLags
    auto cov_ln = [&](int i, int j) {
        const int lo = i < j ? i : j, l = i < j ? j - i : i - j;
        if (l >= kCiLags) return 0.0;
        return bias * h[(size_t)l * nm + lo] / (4.0 * n * n * P[i] * P[j]);
    };
    // f = A ln P (two entries per row), theta = (D + a) f + const
    const double dT = (double)e->spacing, a = (double)e->p.a;
    std::vector<std::vector<std::pair<int, double>>> A(nm), Th(nm);
    for (int m = 0; m < nm; ++m) {
        const int first = (m == 0) ? 0 : m - 1, last = (m == nm - 1) ? nm - 1 : m + 1;
        const double c = -(((m == 0) || (m == nm - 1)) ? 1.0 : 0.5) / dT;
        A[m] = {{last, c}, {first, -c}};
    }
    auto add_row = [&](std::vector<std::pair<int, double>>& dst, const std::vector<std::pair<int, double>>& src, double w) {
        for (const auto& kv : src) {
            bool found = false;
            for (auto& d : dst)
                if (d.first == kv.first) { d.second += w * kv.second; found = true; break; }
            if (!found) dst.push_back({kv.first, w * kv.second});
        }
    };
    for (int i = 0; i < nm; ++i) {
        if (i == 0) { add_row(Th[i], A[1], 1.0 / dT); add_row(Th[i], A[0], -1.0 / dT); }
        else if (i == nm - 1) { add_row(Th[i], A[i], 1.0 / dT); add_row(Th[i], A[i - 1], -1.0 / dT); }
        else { add_row(Th[i], A[i + 1], 0.5 / dT); add_row(Th[i], A[i - 1], -0.5 / dT); }
        add_row(Th[i], A[i], a);
    }
    auto var_of = [&](const std::vector<std::pair<int, double>>& row) {
        double v = 0.0;
        for (const auto& x : row)
            for (const auto& y : row) v += x.second * y.second * cov_ln(x.first, y.first);
        return v > 0.0 ? v : 0.0;
    };
    for (int m = 0; m < nm; ++m) {
        if (f_se) f_se[m] = (float)sqrt(var_of(A[m]));
        if (theta_se) theta_se[m] = (float)sqrt(var_of(Th[m]));
        if (P_se_batch) P_se_batch[m] = (float)(P[m] * sqrt(cov_ln(m, m) > 0 ? cov_ln(m, m) : 0.0));
    }
    return HW1F_OK;
}

// ---- Q2a ----------------------------------------------------------------------------------------
int hw1f_theta_calibrate(hw1f_engine* e, const float* f, float* theta_rec, float* theta_ref, float* T)
{
    HW_TRY(require_model(e));
    if (!f || !theta_rec || !theta_ref || !T) return HW1F_ERR_INVALID;
    HW_CUDA(e, cudaSetDevice(e->device));
    const int n = e->p.n_mat;
    HW_CUDA(e, e->d_out.ensure(4 * (size_t)n));
    float* d_f = e->d_out.p;
    HW_TRY(upload(e, d_f, f, n * sizeof(float)));
    theta_kernel<<<1, n, 0, e->stream>>>(d_f, n, e->p.a, e->p.sigma, e->spacing, e->p.theta_a0, e->p.theta_b0,
                                         e->p.theta_a1, e->p.theta_b1, e->p.theta_break, d_f + n, d_f + 2 * n,
                                         d_f + 3 * n);
    HW_TRY(check_launch(e, "theta_kernel"));
    std::vector<float> host(3 * (size_t)n);
    HW_TRY(download(e, host.data(), d_f + n, host.size() * sizeof(float)));
    memcpy(theta_rec, host.data(), n * sizeof(float));
    memcpy(theta_ref, host.data() + n, n * sizeof(float));
    memcpy(T, host.data() + 2 * n, n * sizeof(float));
    return HW1F_OK;
}

// ---- Q2b ----------------------------------------------------------------------------------------
static int zbc_run(hw1f_engine* e, hw1f_rng* rng, float S1, float S2, float K, const float* P_mkt, const float* f_mkt,
                   int32_t n, double* d_moments, const Finish& fin)
{
    const ScenDev sc = scen_dev(e, e->p.sigma, e->sig_st, 0);
    // the bond plan rides on the jump-table launch (its extra block)
    const PlanJob job = plan_job_host(e, &sc, 1, S1, S2, P_mkt, f_mkt);
    Launch L;
    HW_TRY(prepare_launch(e, &rng->seed, 1, rng->first_path, rng->n_paths, rng->offset, &L, &job));
    HW_TRY(launch_zbc(e, L, &sc, 1, n, K, d_moments, fin));
    rng->offset += (uint64_t)n;
    return HW1F_OK;
}

int hw1f_zbc_cv_moments(hw1f_engine* e, hw1f_rng* rng, float S1, float S2, float K, const float* P_mkt,
                        const float* f_mkt, int32_t n_steps_S1, double* d_moments)
{
    HW_TRY(require_model(e));
    if (!rng || !P_mkt || !f_mkt || !d_moments) return HW1F_ERR_INVALID;
    HW_CUDA(e, cudaSetDevice(e->device));
    int32_t n = 0;
    HW_TRY(resolve_steps(e, S1, n_steps_S1, &n));
    Finish fin;
    fin.exchange = true;
    return zbc_run(e, rng, S1, S2, K, P_mkt, f_mkt, n, d_moments, fin);
}

int hw1f_zbc_cv_finish(hw1f_engine* e, const double* d_moments, uint64_t n_paths_total, float P0S2,
                       hw1f_zbc_result* out)
{
    HW_TRY(require_model(e));
    if (!d_moments || !out) return HW1F_ERR_INVALID;
    HW_REQUIRE(e, n_paths_total >= 1 && n_paths_total < (1ull << 40), "n_paths_total outside [1, 2^40)");
    HW_CUDA(e, cudaSetDevice(e->device));
    double mom[5];
    HW_TRY(download(e, mom, d_moments, sizeof(mom)));
    HW_TRY(require_finite(e, mom, 5));
    zbc_algebra(mom, n_paths_total, P0S2, 0, out);   // the step count is not part of the moments
    return HW1F_OK;
}

int hw1f_zbc_cv(hw1f_engine* e, hw1f_rng* rng, float S1, float S2, float K, const float* P_mkt, const float* f_mkt,
                int32_t n_steps_S1, hw1f_zbc_result* out, float* sim_ms)
{
    HW_TRY(require_model(e));
    if (!rng || !out || !P_mkt || !f_mkt) return HW1F_ERR_INVALID;
    HW_CUDA(e, cudaSetDevice(e->device));
    int32_t n = 0;
    HW_TRY(resolve_steps(e, S1, n_steps_S1, &n));
    HW_CUDA(e, e->d_moments.ensure(4 * (size_t)e->p.n_mat * kMaxRuns));
    HW_TRY(warm_geometry(e, rng));
    Finish fin;
    fin.host_mom = res_mom(e, 0);
    if (sim_ms) HW_CUDA(e, cudaEventRecord(e->ev0, e->stream));
    HW_TRY(zbc_run(e, rng, S1, S2, K, P_mkt, f_mkt, n, e->d_moments.p, fin));
    if (sim_ms) HW_CUDA(e, cudaEventRecord(e->ev1, e->stream));
    HW_TRY(wait_results(e));
    double mom[5];
    memcpy(mom, res_mom(e, 0), sizeof(mom));
    HW_TRY(require_finite(e, mom, 5));
    zbc_algebra(mom, rng->n_paths, P_mkt[e->p.n_mat - 1], n, out);
    if (sim_ms) HW_CUDA(e, cudaEventElapsedTime(sim_ms, e->ev0, e->ev1));
    return HW1F_OK;
}

int hw1f_zbc_cv_batch(hw1f_engine* e, const uint64_t* seeds, int32_t n_runs, uint64_t n_paths, float S1, float S2,
                      float K, const float* P_mkt, const float* f_mkt, int32_t n_steps_S1, hw1f_zbc_result* out,
                      float* sim_ms)
{
    HW_TRY(require_model(e));
    if (!seeds || !out || !P_mkt || !f_mkt) return HW1F_ERR_INVALID;
    HW_REQUIRE(e, 2 * n_paths < (1ull << 31), "the reference's int N_total needs 2*n_paths < 2^31");
    HW_CUDA(e, cudaSetDevice(e->device));
    int32_t n = 0;
    HW_TRY(resolve_steps(e, S1, n_steps_S1, &n));
    HW_CUDA(e, e->d_moments.ensure(4 * (size_t)e->p.n_mat * kMaxRuns));
    const ScenDev sc = scen_dev(e, e->p.sigma, e->sig_st, 0);
    const PlanJob job = plan_job_host(e, &sc, 1, S1, S2, P_mkt, f_mkt);
    {
        const hw1f_rng geom{0, 0, n_paths, 0};
        HW_TRY(warm_geometry(e, &geom));
    }
    HW_CUDA(e, cudaEventRecord(e->ev0, e->stream));
    for (int32_t done = 0; done < n_runs; done += kMaxRuns) {
        const int nb = (n_runs - done < kMaxRuns) ? (n_runs - done) : kMaxRuns;
        Launch L;
        HW_TRY(prepare_launch(e, seeds + done, nb, 0, n_paths, 0, &L, &job));
        Finish fin;
        fin.host_mom = res_mom(e, 0);   // [run][5]
        HW_TRY(launch_zbc(e, L, &sc, 1, n, K, e->d_moments.p, fin));
        HW_TRY(wait_results(e));
        const double* mom = res_mom(e, 0);
        for (int r = 0; r < nb; ++r) zbc_algebra(&mom[5 * r], n_paths, P_mkt[e->p.n_mat - 1], n, &out[done + r]);
    }
    HW_CUDA(e, cudaEventRecord(e->ev1, e->stream));
    HW_CUDA(e, cudaEventSynchronize(e->ev1));
    if (sim_ms) HW_CUDA(e, cudaEventElapsedTime(sim_ms, e->ev0, e->ev1));
    return HW1F_OK;
}

// ---- Q3 ----------------------------------------------------------------------------------------
static int pathwise_run(hw1f_engine* e, hw1f_rng* rng, float S1, float S2, float K, const float* P_mkt,
                        const float* f_mkt, int32_t n, double* d_moments, const Finish& fin)
{
    const ScenDev sc = scen_dev(e, e->p.sigma, e->sig_st, 0);
    const PlanJob job = plan_job_host(e, &sc, 1, S1, S2, P_mkt, f_mkt);
    Launch L;
    HW_TRY(prepare_launch(e, &rng->seed, 1, rng->first_path, rng->n_paths, rng->offset, &L, &job));
    HW_TRY(launch_pathwise(e, L, sc, n, K, d_moments, fin));
    rng->offset += (uint64_t)n;
    return HW1F_OK;
}

int hw1f_vega_pathwise_moments(hw1f_engine* e, hw1f_rng* rng, float S1, float S2, float K, const float* P_mkt,
                               const float* f_mkt, int32_t n_steps_S1, double* d_moments)
{
    HW_TRY(require_model(e));
    if (!rng || !P_mkt || !f_mkt || !d_moments) return HW1F_ERR_INVALID;
    HW_CUDA(e, cudaSetDevice(e->device));
    int32_t n = 0;
    HW_TRY(resolve_steps(e, S1, n_steps_S1, &n));
    Finish fin;
    fin.exchange = true;
    return pathwise_run(e, rng, S1, S2, K, P_mkt, f_mkt, n, d_moments, fin);
}

static void pathwise_result(const double mom[2], uint64_t n_paths, hw1f_vega_result* out)
{
    const double np = (double)n_paths;
    out->vega_pathwise = (float)mom[0] / (float)n_paths;   // sum / N_PATHS in float, src/3:261
    out->vega_pathwise_f64 = mom[0] / np;
    const double var = (np > 1) ? (mom[1] - mom[0] * mom[0] / np) / (np - 1.0) : 0.0;
    out->vega_pathwise_se = (var > 0) ? sqrt(var / np) : 0.0;
}

int hw1f_vega_pathwise(hw1f_engine* e, hw1f_rng* rng, float S1, float S2, float K, const float* P_mkt,
                       const float* f_mkt, int32_t n_steps_S1, hw1f_vega_result* out)
{
    HW_TRY(require_model(e));
    if (!rng || !out || !P_mkt || !f_mkt) return HW1F_ERR_INVALID;
    HW_CUDA(e, cudaSetDevice(e->device));
    int32_t n = 0;
    HW_TRY(resolve_steps(e, S1, n_steps_S1, &n));
    HW_CUDA(e, e->d_moments.ensure(4 * (size_t)e->p.n_mat * kMaxRuns));
    HW_TRY(warm_geometry(e, rng));
    Finish fin;
    fin.host_mom = res_mom(e, 0);
    HW_CUDA(e, cudaEventRecord(e->ev0, e->stream));
    HW_TRY(pathwise_run(e, rng, S1, S2, K, P_mkt, f_mkt, n, e->d_moments.p, fin));
    HW_CUDA(e, cudaEventRecord(e->ev1, e->stream));
    HW_TRY(wait_results(e));
    double mom[2];
    memcpy(mom, res_mom(e, 0), sizeof(mom));
    HW_TRY(require_finite(e, mom, 2));
    out->n_steps_S1 = n;
    pathwise_result(mom, rng->n_paths, out);
    HW_CUDA(e, cudaEventElapsedTime(&out->ms_pathwise, e->ev0, e->ev1));
    return HW1F_OK;
}

int hw1f_vega_pathwise_batch(hw1f_engine* e, const uint64_t* seeds, int32_t n_runs, uint64_t n_paths, float S1,
                             float S2, float K, const float* P_mkt, const float* f_mkt, int32_t n_steps_S1,
                             float* vega, float* sim_ms)
{
    HW_TRY(require_model(e));
    if (!seeds || !vega || !P_mkt || !f_mkt) return HW1F_ERR_INVALID;
    HW_CUDA(e, cudaSetDevice(e->device));
    int32_t n = 0;
    HW_TRY(resolve_steps(e, S1, n_steps_S1, &n));
    HW_CUDA(e, e->d_moments.ensure(4 * (size_t)e->p.n_mat * kMaxRuns));
    const ScenDev sc = scen_dev(e, e->p.sigma, e->sig_st, 0);
    const PlanJob job = plan_job_host(e, &sc, 1, S1, S2, P_mkt, f_mkt);
    {
        const hw1f_rng geom{0, 0, n_paths, 0};
        HW_TRY(warm_geometry(e, &geom));
    }
    HW_CUDA(e, cudaEventRecord(e->ev0, e->stream));
    for (int32_t done = 0; done < n_runs; done += kMaxRuns) {
        const int nb = (n_runs - done < kMaxRuns) ? (n_runs - done) : kMaxRuns;
        Launch L;
        HW_TRY(prepare_launch(e, seeds + done, nb, 0, n_paths, 0, &L, &job));
        Finish fin;
        fin.host_mom = res_mom(e, 0);   // [run][2]
        HW_TRY(launch_pathwise(e, L, sc, n, K, e->d_moments.p, fin));
        HW_TRY(wait_results(e));
        const double* mom = res_mom(e, 0);
        for (int r = 0; r < nb; ++r) vega[done + r] = (float)mom[2 * r] / (float)n_paths;   // src/3:561
    }
    HW_CUDA(e, cudaEventRecord(e->ev1, e->stream));
    HW_CUDA(e, cudaEventSynchronize(e->ev1));
    if (sim_ms) HW_CUDA(e, cudaEventElapsedTime(sim_ms, e->ev0, e->ev1));
    return HW1F_OK;
}

// CV-adjusted price of run_zbc_price (src/3:110-166) from five double moments
static float zbc_price_cv(const double mom[5], uint64_t n_paths, float P0S2)
{
    hw1f_zbc_result r;
    zbc_algebra(mom, n_paths, P0S2, 0, &r);
    return r.price_cv;
}

// run_finite_difference, src/3:400-446: sigma -/+ eps, sig_st and shifted drift per bump; both bumps read the same
// market curves and the same normals.  ONE jump-table launch (with both bond plans) + ONE simulation launch.
static int fd_run(hw1f_engine* e, hw1f_rng* rng, float S1, float S2, float K, const float* P_mkt, const float* f_mkt,
                  float eps, int32_t n, double* d_moments, const Finish& fin)
{
    const float sig_m = e->p.sigma - eps, sig_p = e->p.sigma + eps;
    HW_TRY(upload_fd_tables(e, sig_m, sig_p));
    ScenDev sc[2] = {scen_dev(e, sig_m, host_sig_st(e->p, sig_m), 2), scen_dev(e, sig_p, host_sig_st(e->p, sig_p), 3)};
    const PlanJob job = plan_job_host(e, sc, 2, S1, S2, P_mkt, f_mkt);
    Launch L;
    HW_TRY(prepare_launch(e, &rng->seed, 1, rng->first_path, rng->n_paths, rng->offset, &L, &job));
    HW_TRY(launch_zbc(e, L, sc, 2, n, K, d_moments, fin));
    rng->offset += (uint64_t)n;
    return HW1F_OK;
}

// run_finite_difference_recalibrated, src/3:484-525.  recompute_market_data (src/3:449-482) re-simulates the curve at
// sigma -/+ eps with the UNSHIFTED base drift (compute_drift_tables only changes the sensitivity table) on normals
// [off, off+N_STEPS); the prices then reuse normals [off, off+n) with the recalibrated curves, base drift, bumped
// sig_st and sigma.  Decomposed mode, S1 on the maturity grid: the curve pass parks every subsequence's noise state at
// step n, its LAST BLOCK reduces, finalises both curves on the device and computes their bond plans, and the two
// prices are evaluated from the parked state -- normals [off, off+n) are the first n normals of the curve window, so
// nothing is simulated twice (8 bytes of state per subsequence: above 2^27 subsequences the second pass is used).
// res_area: curves (P0S2 of both) and the ten price moments land in that result area.
static int recal_run(hw1f_engine* e, hw1f_rng* rng, float S1, float S2, float K, float eps, int32_t n, double* d_moments,
                     int res_area)
{
    const float sig_m = e->p.sigma - eps, sig_p = e->p.sigma + eps;
    ScenDev sc[2] = {scen_dev(e, sig_m, host_sig_st(e->p, sig_m), 0), scen_dev(e, sig_p, host_sig_st(e->p, sig_p), 0)};
    Launch L;
    HW_TRY(prepare_launch(e, &rng->seed, 1, rng->first_path, rng->n_paths, rng->offset, &L));
    const bool one_pass = e->mode == HW1F_MODE_DECOMPOSED && n > 0 && (e->stride & 1) == 0 && (n % e->stride) == 0 &&
                          rng->n_paths <= (1ull << 27);
    Finish fc;
    fc.epi = true;
    fc.n_total = rng->n_paths;
    fc.dev_curve = e->d_mkt.p;
    fc.host_curve = res_curve(e, res_area);
    fc.plan = plan_job_dev(e, sc, 2, S1, S2);
    HW_TRY(launch_curve(e, L, sc, 2, e->d_moments.p, one_pass ? n : 0, fc, one_pass ? keep_code(e, S1, S2) : 0));
    Finish fz;
    fz.host_mom = res_mom(e, res_area);
    if (one_pass) HW_TRY(launch_zbc_from_state(e, L, sc, n, K, d_moments, fz));
    else HW_TRY(launch_zbc(e, L, sc, 2, n, K, d_moments, fz));
    rng->offset += (uint64_t)n;   // the reference leaves d_states after run_zbc_price (src/3:509-510)
    return HW1F_OK;
}

static void recal_result(hw1f_engine* e, int res_area, uint64_t n_paths, float eps, hw1f_vega_result* out)
{
    const int nm = e->p.n_mat;
    const double* mom = res_mom(e, res_area);
    const float* cur = res_curve(e, res_area);
    const float P0S2[2] = {cur[nm - 1], cur[3 * (size_t)nm + nm - 1]};
    out->price_minus_recal = zbc_price_cv(mom, n_paths, P0S2[0]);
    out->price_plus_recal = zbc_price_cv(mom + 5, n_paths, P0S2[1]);
    out->vega_fd_recal = (out->price_plus_recal - out->price_minus_recal) / (2.0f * eps);   // src/3:513
}

int hw1f_vega_fd(hw1f_engine* e, hw1f_rng* rng, float S1, float S2, float K, const float* P_mkt, const float* f_mkt,
                 float eps, int32_t n_steps_S1, hw1f_vega_result* out)
{
    HW_TRY(require_model(e));
    if (!rng || !out || !P_mkt || !f_mkt) return HW1F_ERR_INVALID;
    HW_REQUIRE(e, 2 * rng->n_paths < (1ull << 31), "the reference's int N_total needs 2*n_paths < 2^31");
    HW_CUDA(e, cudaSetDevice(e->device));
    int32_t n = 0;
    HW_TRY(resolve_steps(e, S1, n_steps_S1, &n));
    HW_CUDA(e, e->d_moments.ensure(4 * (size_t)e->p.n_mat * kMaxRuns));
    HW_TRY(warm_geometry(e, rng));
    Finish fin;
    fin.host_mom = res_mom(e, 0);
    HW_CUDA(e, cudaEventRecord(e->ev0, e->stream));
    HW_TRY(fd_run(e, rng, S1, S2, K, P_mkt, f_mkt, eps, n, e->d_moments.p, fin));
    HW_CUDA(e, cudaEventRecord(e->ev1, e->stream));
    HW_TRY(wait_results(e));
    double mom[10];
    memcpy(mom, res_mom(e, 0), sizeof(mom));
    HW_TRY(require_finite(e, mom, 10));
    const float P0S2 = P_mkt[e->p.n_mat - 1];
    out->n_steps_S1 = n;
    out->price_minus = zbc_price_cv(mom, rng->n_paths, P0S2);
    out->price_plus = zbc_price_cv(mom + 5, rng->n_paths, P0S2);
    out->vega_fd = (out->price_plus - out->price_minus) / (2.0f * eps);   // src/3:443
    HW_CUDA(e, cudaEventElapsedTime(&out->ms_fd, e->ev0, e->ev1));
    return HW1F_OK;
}

int hw1f_vega_fd_recalibrated(hw1f_engine* e, hw1f_rng* rng, float S1, float S2, float K, float eps,
                              int32_t n_steps_S1, hw1f_vega_result* out)
{
    HW_TRY(require_model(e));
    if (!rng || !out) return HW1F_ERR_INVALID;
    HW_REQUIRE(e, 2 * rng->n_paths < (1ull << 31), "the reference's int N_total needs 2*n_paths < 2^31");
    HW_CUDA(e, cudaSetDevice(e->device));
    if (rng->offset & 1) {
        e->err = "recalibrated FD needs an even normal offset (its curve window starts on a Box-Muller pair boundary)";
        return HW1F_ERR_UNSUPPORTED;
    }
    int32_t n = 0;
    HW_TRY(resolve_steps(e, S1, n_steps_S1, &n));
    const int nm = e->p.n_mat;
    HW_CUDA(e, e->d_moments.ensure(4 * (size_t)nm * kMaxRuns));
    HW_CUDA(e, e->d_mkt.ensure(4 * (size_t)nm));
    HW_TRY(warm_geometry(e, rng));
    HW_CUDA(e, cudaEventRecord(e->ev0, e->stream));
    HW_TRY(recal_run(e, rng, S1, S2, K, eps, n, e->d_moments.p + 4 * (size_t)nm, 0));
    HW_CUDA(e, cudaEventRecord(e->ev1, e->stream));
    HW_TRY(wait_results(e));
    HW_TRY(require_finite(e, res_mom(e, 0), 10));
    out->n_steps_S1 = n;
    recal_result(e, 0, rng->n_paths, eps, out);
    HW_CUDA(e, cudaEventElapsedTime(&out->ms_fd_recal, e->ev0, e->ev1));
    return HW1F_OK;
}

int hw1f_vega(hw1f_engine* e, hw1f_rng* rng, float S1, float S2, float K, const float* P_mkt, const float* f_mkt,
              float eps, int32_t n_steps_S1, hw1f_vega_result* out)
{
    HW_TRY(require_model(e));
    if (!rng || !out || !P_mkt || !f_mkt) return HW1F_ERR_INVALID;
    HW_REQUIRE(e, 2 * rng->n_paths < (1ull << 31), "the reference's int N_total needs 2*n_paths < 2^31");
    HW_CUDA(e, cudaSetDevice(e->device));
    memset(out, 0, sizeof(*out));
    int32_t n = 0;
    HW_TRY(resolve_steps(e, S1, n_steps_S1, &n));
    const int nm = e->p.n_mat;
    if ((rng->offset & 1) || (e->stride & 1)) {
        // the recalibration window [off+2n, ..) must start on a Box-Muller pair boundary: take the three calls, whose
        // own checks report what is unsupported
        HW_TRY(hw1f_vega_pathwise(e, rng, S1, S2, K, P_mkt, f_mkt, n, out));     // normals [0,n)
        HW_TRY(hw1f_vega_fd(e, rng, S1, S2, K, P_mkt, f_mkt, eps, n, out));      // normals [n,2n)
        return hw1f_vega_fd_recalibrated(e, rng, S1, S2, K, eps, n, out);        // normals [2n,..)
    }
    const bool one_launch = e->mode == HW1F_MODE_DECOMPOSED && n > 0 && (n & 1) == 0 && (e->stride & 1) == 0 && (n % e->stride) == 0 &&
                            rng->n_paths <= (1ull << 27) && e->seq_one_launch;
    if (one_launch) {
        // ONE pass over each subsequence's normals (fast_kernel SEQ): pathwise tangent on [off, off+n), both CRN bumps on
        // [off+n, off+2n), the two recalibration curves on [off+2n, off+2n+N_STEPS) with the noise state parked at step
        // n of that window; the tail kernel reduces, finalises both recalibrated curves and their bond plans; the two
        // recalibrated prices come from the parked state.  Five launches (jump table, simulation, tail, prices, tail)
        // instead of eleven, one stream derivation per subsequence instead of three.  Same draw windows, same results.
        HW_CUDA(e, e->d_moments.ensure(4 * (size_t)nm * kMaxRuns));
        HW_CUDA(e, e->d_mkt.ensure(4 * (size_t)nm));
        const float sig_m = e->p.sigma - eps, sig_p = e->p.sigma + eps;
        HW_TRY(upload_fd_tables(e, sig_m, sig_p));
        const ScenDev base = scen_dev(e, e->p.sigma, e->sig_st, 0);
        const ScenDev three[3] = {base, scen_dev(e, sig_m, host_sig_st(e->p, sig_m), 2),
                                  scen_dev(e, sig_p, host_sig_st(e->p, sig_p), 3)};
        ScenDev rc[2] = {scen_dev(e, sig_m, host_sig_st(e->p, sig_m), 0), scen_dev(e, sig_p, host_sig_st(e->p, sig_p), 0)};
        HW_TRY(warm_geometry(e, rng));
        HW_CUDA(e, cudaEventRecord(e->ev0, e->stream));
        const PlanJob job = plan_job_host(e, three, 3, S1, S2, P_mkt, f_mkt);
        Launch L;
        HW_TRY(prepare_launch(e, &rng->seed, 1, rng->first_path, rng->n_paths, rng->offset, &L, &job));
        const int nq = 4 * nm + 18;
        HW_CUDA(e, e->d_partials.ensure((size_t)L.grid_x * nq));
        HW_CUDA(e, e->d_state.ensure((size_t)L.g.n_chunks * kChunk));
        const FastScen c0 = fast_scen(e, rc[0].sig_st, 0, 0), c1 = fast_scen(e, rc[1].sig_st, 0, 0);
        const FastScen zb = fast_scen(e, base.sig_st, 0, n), zm = fast_scen(e, three[1].sig_st, 2, n),
                       zp = fast_scen(e, three[2].sig_st, 3, n);
        const FastTangent tg = fast_tangent(e, n);
        const size_t smem = smem_fast(e, 2, 3, 1, 1);
        HW_TRY(set_smem(e, (fast_kernel<2, 3, 1, 1, 1>), smem));
        HW_CUDA(e, launch_k(fast_kernel<2, 3, 1, 1, 1>, dim3(L.grid_x), kThreads, smem, e->stream, true, L.g, L.seeds,
                            model_dev(e), c0, c1, zb, zm, zp, tg, e->d_plans.p, n, keep_code(e, S1, S2), K, e->d_partials.p,
                            e->d_state.p));
        HW_TRY(check_launch(e, "fast_kernel<q3 sequence>"));
        Finish fc;
        fc.host_mom = res_mom(e, 0);          // [4 nm curve sums][5 unused][pathwise 3][FD- 5][FD+ 5]
        fc.epi = true;
        fc.n_total = rng->n_paths;
        fc.dev_curve = e->d_mkt.p;
        fc.host_curve = res_curve(e, 0);
        fc.plan = plan_job_dev(e, rc, 2, S1, S2);
        HW_TRY(launch_tail(e, L, L.g.n_paths, nq, 2, c0.emI, c1.emI, 2.0f, e->d_moments.p, nq, 18, fc));
        Finish fz;
        fz.host_mom = res_mom(e, 1);
        HW_TRY(launch_zbc_from_state(e, L, rc, n, K, e->d_moments.p + nq, fz));
        HW_CUDA(e, cudaEventRecord(e->ev1, e->stream));
        rng->offset += 3 * (uint64_t)n;
        HW_TRY(wait_results(e));
        const double* ext = res_mom(e, 0) + 4 * (size_t)nm;
        HW_TRY(require_finite(e, ext, 18));
        HW_TRY(require_finite(e, res_mom(e, 1), 10));
        const float P0S2 = P_mkt[nm - 1];
        out->n_steps_S1 = n;
        pathwise_result(ext + 5, rng->n_paths, out);
        out->price_minus = zbc_price_cv(ext + 8, rng->n_paths, P0S2);
        out->price_plus = zbc_price_cv(ext + 13, rng->n_paths, P0S2);
        out->vega_fd = (out->price_plus - out->price_minus) / (2.0f * eps);                     // src/3:443
        {
            const float* cur = res_curve(e, 0);
            const float P0S2_rc[2] = {cur[nm - 1], cur[3 * (size_t)nm + nm - 1]};
            out->price_minus_recal = zbc_price_cv(res_mom(e, 1), rng->n_paths, P0S2_rc[0]);
            out->price_plus_recal = zbc_price_cv(res_mom(e, 1) + 5, rng->n_paths, P0S2_rc[1]);
            out->vega_fd_recal = (out->price_plus_recal - out->price_minus_recal) / (2.0f * eps);   // src/3:513
        }
        float ms = 0.f;   // one launch: apportioned by the normals each estimator consumed
        HW_CUDA(e, cudaEventElapsedTime(&ms, e->ev0, e->ev1));
        const float tot = (float)(2 * n + e->p.n_steps);
        out->ms_pathwise = ms * (float)n / tot;
        out->ms_fd = ms * (float)n / tot;
        out->ms_fd_recal = ms * (float)e->p.n_steps / tot;
        return HW1F_OK;
    }
    // The three estimators of the reference's main() (src/3:697-834) enqueued back to back -- same draw windows and
    // same results as hw1f_vega_pathwise + hw1f_vega_fd + hw1f_vega_fd_recalibrated -- seven launches in all (three
    // jump tables, three simulations, the prices from the parked state); every result lands in mapped pinned host
    // memory from the kernels' tails, the host waits ONCE.
    HW_CUDA(e, e->d_moments.ensure(4 * (size_t)nm * kMaxRuns));
    HW_CUDA(e, e->d_mkt.ensure(4 * (size_t)nm));
    double* const res = e->d_moments.p + 4 * (size_t)nm;   // [0,2) pathwise, [8,18) FD, [24,34) recalibrated FD
    HW_TRY(warm_geometry(e, rng));
    // pathwise tangent, normals [off, off+n)  (simulate_sensitivity, src/3:251)
    HW_CUDA(e, cudaEventRecord(e->ev0, e->stream));
    Finish f0;
    f0.host_mom = res_mom(e, 0);
    HW_TRY(pathwise_run(e, rng, S1, S2, K, P_mkt, f_mkt, n, res, f0));
    // CRN finite differences, normals [off+n, off+2n)  (run_finite_difference, src/3:400-446)
    HW_CUDA(e, cudaEventRecord(e->ev1, e->stream));
    Finish f1;
    f1.host_mom = res_mom(e, 1);
    HW_TRY(fd_run(e, rng, S1, S2, K, P_mkt, f_mkt, eps, n, res + 8, f1));
    // recalibrated finite differences, curves on [off+2n, off+2n+N_STEPS), prices on [off+2n, off+3n)  (src/3:449-525)
    HW_CUDA(e, cudaEventRecord(e->ev2, e->stream));
    HW_TRY(recal_run(e, rng, S1, S2, K, eps, n, res + 24, 2));
    HW_CUDA(e, cudaEventRecord(e->ev3, e->stream));
    HW_TRY(wait_results(e));
    HW_TRY(require_finite(e, res_mom(e, 0), 2));
    HW_TRY(require_finite(e, res_mom(e, 1), 10));
    HW_TRY(require_finite(e, res_mom(e, 2), 10));
    const float P0S2 = P_mkt[nm - 1];
    out->n_steps_S1 = n;
    pathwise_result(res_mom(e, 0), rng->n_paths, out);
    out->price_minus = zbc_price_cv(res_mom(e, 1), rng->n_paths, P0S2);
    out->price_plus = zbc_price_cv(res_mom(e, 1) + 5, rng->n_paths, P0S2);
    out->vega_fd = (out->price_plus - out->price_minus) / (2.0f * eps);                     // src/3:443
    recal_result(e, 2, rng->n_paths, eps, out);
    HW_CUDA(e, cudaEventElapsedTime(&out->ms_pathwise, e->ev0, e->ev1));
    HW_CUDA(e, cudaEventElapsedTime(&out->ms_fd, e->ev1, e->ev2));
    HW_CUDA(e, cudaEventElapsedTime(&out->ms_fd_recal, e->ev2, e->ev3));
    return HW1F_OK;
}

static int fused_launch(hw1f_engine* e, hw1f_rng* rng, float S1, float S2, float K, const float* P_mkt,
                        const float* f_mkt, bool fd, float eps, int32_t n_steps_S1, double* d_moments, const Finish& fin)
{
    HW_TRY(require_model(e));
    if (!rng || !P_mkt || !f_mkt || !d_moments) return HW1F_ERR_INVALID;
    HW_CUDA(e, cudaSetDevice(e->device));
    int32_t n = 0;
    HW_TRY(resolve_steps(e, S1, n_steps_S1, &n));
    if ((rng->offset & 1) || (e->stride & 1) || n <= 0 || (n % e->stride) != 0) {
        e->err = "fused pass needs an even normal offset, an even save stride and n_steps_S1 on the maturity grid";
        return HW1F_ERR_UNSUPPORTED;
    }
    ScenDev sc[3] = {scen_dev(e, e->p.sigma, e->sig_st, 0), scen_dev(e, e->p.sigma, e->sig_st, 0),
                     scen_dev(e, e->p.sigma, e->sig_st, 0)};
    if (fd) {   // run_finite_difference's scenarios (src/3:414-435): sigma -/+ eps, shifted drift, same curves
        const float sig_m = e->p.sigma - eps, sig_p = e->p.sigma + eps;
        HW_TRY(upload_fd_tables(e, sig_m, sig_p));
        sc[1] = scen_dev(e, sig_m, host_sig_st(e->p, sig_m), 2);
        sc[2] = scen_dev(e, sig_p, host_sig_st(e->p, sig_p), 3);
    }
    // the bond plans (base, and both bumps) ride on the jump-table launch
    const PlanJob job = plan_job_host(e, sc, fd ? 3 : 1, S1, S2, P_mkt, f_mkt);
    Launch L;
    HW_TRY(prepare_launch(e, &rng->seed, 1, rng->first_path, rng->n_paths, rng->offset, &L, &job));
    const int nm = e->p.n_mat, next = kFusedExtra + (fd ? kFusedFdExtra : 0), nq = 2 * nm + next;
    HW_CUDA(e, e->d_partials.ensure((size_t)L.grid_x * nq));
    if (e->mode == HW1F_MODE_DECOMPOSED) {
        // one noise recursion per stream carries the curve, the base ZBC, both bumped ZBCs and both
        // tangent twins; the S1 block comes out in the ABI order [ZBC][vega 3][ZBC-][ZBC+]
        const FastScen c0 = fast_scen(e, sc[0].sig_st, 0, n);
        const FastScen zm = fd ? fast_scen(e, sc[1].sig_st, 2, n) : c0, zp = fd ? fast_scen(e, sc[2].sig_st, 3, n) : c0;
        const FastTangent tg = fast_tangent(e, n);
        const size_t smemf = smem_fast(e, 1, 1, 2);
        const ModelDev md = model_dev(e);
        if (fd) {
            HW_TRY(set_smem(e, fast_kernel<1, 3, 2>, smemf));
            HW_CUDA(e, launch_k(fast_kernel<1, 3, 2>, dim3(L.grid_x), kThreads, smemf, e->stream, true, L.g, L.seeds, md, c0,
                                c0, c0, zm, zp, tg, e->d_plans.p, n, 0, K, e->d_partials.p, (float2*)nullptr));
        } else {
            HW_TRY(set_smem(e, fast_kernel<1, 1, 2>, smemf));
            HW_CUDA(e, launch_k(fast_kernel<1, 1, 2>, dim3(L.grid_x), kThreads, smemf, e->stream, true, L.g, L.seeds, md, c0,
                                c0, c0, c0, c0, tg, e->d_plans.p, n, 0, K, e->d_partials.p, (float2*)nullptr));
        }
        HW_TRY(check_launch(e, "fast_kernel<fused>"));
        HW_TRY(launch_tail(e, L, L.g.n_paths, nq, 1, c0.emI, c0.emI, 2.0f, d_moments, nq, next, fin));
        rng->offset += (uint64_t)e->p.n_steps;
        return HW1F_OK;
    }
    const size_t smem = (size_t)kWinWords * 4 + (size_t)(e->p.n_steps / 2 + (fd ? 3 : 1) * (n / 2)) * sizeof(float4) +
                        (size_t)nq * sizeof(double) + (size_t)kWarps * 2 * nm * sizeof(float) + (size_t)nm * sizeof(float);
    if (fd) {
        HW_TRY(set_smem(e, fused_kernel<true>, smem));
        fused_kernel<true><<<L.grid_x, kThreads, smem, e->stream>>>(L.g, L.seeds, model_dev(e), sc[0], sc[1], sc[2],
                                                                    e->d_plans.p, n, K, e->d_partials.p);
    } else {
        HW_TRY(set_smem(e, fused_kernel<false>, smem));
        fused_kernel<false><<<L.grid_x, kThreads, smem, e->stream>>>(L.g, L.seeds, model_dev(e), sc[0], sc[0], sc[0],
                                                                     e->d_plans.p, n, K, e->d_partials.p);
    }
    HW_TRY(check_launch(e, "fused_kernel"));
    HW_TRY(launch_tail(e, L, L.g.n_paths, nq, 1, sc[0].center, sc[0].center, 1.0f, d_moments, nq, next, fin));
    rng->offset += (uint64_t)e->p.n_steps;
    return HW1F_OK;
}

int hw1f_fused_moments(hw1f_engine* e, hw1f_rng* rng, float S1, float S2, float K, const float* P_mkt,
                       const float* f_mkt, int32_t n_steps_S1, double* d_moments)
{
    if (!e) return HW1F_ERR_INVALID;
    Finish fin;
    fin.exchange = true;
    return fused_launch(e, rng, S1, S2, K, P_mkt, f_mkt, false, 0.0f, n_steps_S1, d_moments, fin);
}

int hw1f_fused_fd_moments(hw1f_engine* e, hw1f_rng* rng, float S1, float S2, float K, const float* P_mkt,
                          const float* f_mkt, float eps, int32_t n_steps_S1, double* d_moments)
{
    if (!e) return HW1F_ERR_INVALID;
    HW_REQUIRE(e, eps > 0.0f && eps < e->p.sigma, "eps must be in (0, sigma)");
    Finish fin;
    fin.exchange = true;
    return fused_launch(e, rng, S1, S2, K, P_mkt, f_mkt, true, eps, n_steps_S1, d_moments, fin);
}

// finalisation of a fused moment vector that sits in the result area (moments from index 2*n_mat on, curves)
static int fused_results(hw1f_engine* e, int area, uint64_t n_paths_total, float P0S2, float eps, int32_t n_steps_S1,
                         float* P, float* f, float* P_se, hw1f_zbc_result* zbc, hw1f_vega_result* vega)
{
    const bool fd = eps > 0.0f;
    const int nm = e->p.n_mat, next = kFusedExtra + (fd ? kFusedFdExtra : 0);
    const double* ext = res_mom(e, area) + 2 * (size_t)nm;
    HW_TRY(require_finite(e, ext, next));
    HW_TRY(read_curve(e, area, 0, P, f, P_se));
    zbc_algebra(ext, n_paths_total, P0S2, n_steps_S1, zbc);
    memset(vega, 0, sizeof(*vega));
    vega->n_steps_S1 = n_steps_S1;
    const double np2 = 2.0 * (double)n_paths_total, np1 = (double)n_paths_total;
    vega->vega_pathwise_f64 = ext[5] / np2;                 // both antithetic twins
    vega->vega_pathwise = (float)vega->vega_pathwise_f64;
    const double mean_pair = ext[5] / np1;                  // pair sums: var of the pair mean
    const double var_pair = (np1 > 1) ? (ext[6] - np1 * mean_pair * mean_pair) / (np1 - 1.0) : 0.0;
    vega->vega_pathwise_se = (var_pair > 0) ? 0.5 * sqrt(var_pair / np1) : 0.0;
    if (fd) {
        vega->price_minus = zbc_price_cv(ext + kFusedExtra, n_paths_total, P0S2);
        vega->price_plus = zbc_price_cv(ext + kFusedExtra + 5, n_paths_total, P0S2);
        vega->vega_fd = (vega->price_plus - vega->price_minus) / (2.0f * eps);
    }
    return HW1F_OK;
}

int hw1f_fused_finish(hw1f_engine* e, const double* d_moments, uint64_t n_paths_total, float P0S2, float eps,
                      int32_t n_steps_S1, float* P, float* f, float* P_se, hw1f_zbc_result* zbc, hw1f_vega_result* vega)
{
    HW_TRY(require_model(e));
    if (!d_moments || !P || !f || !zbc || !vega) return HW1F_ERR_INVALID;
    HW_CUDA(e, cudaSetDevice(e->device));
    HW_REQUIRE(e, n_paths_total >= 1 && n_paths_total < (1ull << 40), "n_paths_total outside [1, 2^40)");
    const int nm = e->p.n_mat, next = kFusedExtra + (eps > 0.0f ? kFusedFdExtra : 0);
    // curve epilogue on the device and the whole vector into the result area: one launch, one wait
    Finish fin;
    fin.host_mom = res_mom(e, 0);
    fin.epi = true;
    fin.n_total = n_paths_total;
    fin.host_curve = res_curve(e, 0);
    HW_TRY(publish(e, 1, 1, const_cast<double*>(d_moments), 2 * nm + next, next, fin));
    HW_TRY(wait_results(e));
    return fused_results(e, 0, n_paths_total, P0S2, eps, n_steps_S1, P, f, P_se, zbc, vega);
}

int hw1f_fused(hw1f_engine* e, hw1f_rng* rng, float S1, float S2, float K, const float* P_mkt, const float* f_mkt,
               float eps, int32_t n_steps_S1, float* P, float* f, float* P_se, hw1f_zbc_result* zbc,
               hw1f_vega_result* vega, float* sim_ms)
{
    HW_TRY(require_model(e));
    if (!rng || !P_mkt || !f_mkt || !P || !f || !zbc || !vega) return HW1F_ERR_INVALID;
    HW_REQUIRE(e, eps > 0.0f, "hw1f_fused needs eps > 0 (the FD bumps ride on the same launch)");
    HW_CUDA(e, cudaSetDevice(e->device));
    int32_t n = 0;
    HW_TRY(resolve_steps(e, S1, n_steps_S1, &n));
    const int nm = e->p.n_mat;
    HW_CUDA(e, e->d_moments.ensure(4 * (size_t)nm * kMaxRuns));
    HW_TRY(warm_geometry(e, rng));
    Finish fin;
    fin.host_mom = res_mom(e, 0);
    fin.epi = true;
    fin.n_total = rng->n_paths;
    fin.host_curve = res_curve(e, 0);
    HW_CUDA(e, cudaEventRecord(e->ev0, e->stream));
    HW_TRY(fused_launch(e, rng, S1, S2, K, P_mkt, f_mkt, true, eps, n, e->d_moments.p, fin));
    HW_CUDA(e, cudaEventRecord(e->ev1, e->stream));
    HW_TRY(wait_results(e));
    HW_TRY(fused_results(e, 0, rng->n_paths, P_mkt[nm - 1], eps, n, P, f, P_se, zbc, vega));
    float ms = 0.f;
    HW_CUDA(e, cudaEventElapsedTime(&ms, e->ev0, e->ev1));
    vega->ms_pathwise = vega->ms_fd = ms;
    if (sim_ms) *sim_ms = ms;
    return HW1F_OK;
}

// ---- caps and floors ------------------------------------------------------------------------------
// every argument checked before any launch; steps[i] = the resolved reset step of caplet i
static int cap_validate(hw1f_engine* e, int32_t kind, const hw1f_caplet* caps, int32_t n, std::vector<int>& steps)
{
    HW_REQUIRE(e, kind == HW1F_KIND_CAP || kind == HW1F_KIND_FLOOR, "kind must be HW1F_KIND_CAP or HW1F_KIND_FLOOR");
    HW_REQUIRE(e, n >= 1 && n <= HW1F_MAX_CAPLETS, "n_caplets must be in [1, HW1F_MAX_CAPLETS]");
    steps.assign(n, 0);
    const double dt = (double)e->dt;
    for (int i = 0; i < n; ++i) {
        const hw1f_caplet& c = caps[i];
        const std::string at = " (caplet " + std::to_string(i) + ")";
        HW_REQUIRE(e, std::isfinite(c.T_reset) && c.T_reset > 0.0f, "T_reset must be finite and positive" + at);
        HW_REQUIRE(e, std::isfinite(c.T_pay) && c.T_pay > c.T_reset, "T_pay must be greater than T_reset" + at);
        HW_REQUIRE(e, c.T_pay <= e->p.T_final, "T_pay must not exceed T_final" + at);
        HW_REQUIRE(e, std::isfinite(c.K) && c.K > 0.0f, "K must be finite and positive" + at);
        HW_REQUIRE(e, std::isfinite(c.N) && c.N > 0.0f, "N must be finite and positive" + at);
        long k = c.n_steps_reset;
        if (k < 0) {
            // nearest step, not truncation: a date a hair below a step must not move the reset by a whole step
            k = std::lround((double)c.T_reset / dt);
            HW_REQUIRE(e, std::fabs((double)c.T_reset - (double)k * dt) <= 1e-3 * dt,
                       "T_reset is not on the step grid (|T_reset - k dt| > 1e-3 dt): pass n_steps_reset" + at);
        }
        HW_REQUIRE(e, k >= 1 && k <= e->p.n_steps, "reset step outside [1, n_steps]" + at);
        HW_REQUIRE(e, i == 0 || k >= steps[i - 1], "reset steps must be non-decreasing along the strip" + at);
        steps[i] = (int)k;
    }
    return HW1F_OK;
}

// one staged upload of [caplet table | P_mkt | f_mkt], the launch and its tail
static int cap_run(hw1f_engine* e, hw1f_rng* rng, int32_t kind, const hw1f_caplet* caps, int32_t n,
                   const std::vector<int>& steps, const float* P_mkt, const float* f_mkt, double* d_moments,
                   const Finish& fin)
{
    const int nm = e->p.n_mat, nq = 5 * (n + 1);
    const size_t tab = ((size_t)n * sizeof(CapletDev) + 255) & ~(size_t)255;
    std::vector<char> h(tab + 2 * (size_t)nm * sizeof(float), 0);
    CapletDev* cd = reinterpret_cast<CapletDev*>(h.data());
    for (int i = 0; i < n; ++i) {
        cd[i].T_reset = caps[i].T_reset;
        cd[i].T_pay = caps[i].T_pay;
        cd[i].K = caps[i].K;
        cd[i].N = caps[i].N;
        cd[i].m = (float)e->det_m[0][steps[i]];
        cd[i].Im = (float)e->det_I[0][steps[i]];
        cd[i].step = steps[i];
        cd[i].pad = 0;
    }
    memcpy(h.data() + tab, P_mkt, nm * sizeof(float));
    memcpy(h.data() + tab + nm * sizeof(float), f_mkt, nm * sizeof(float));
    const int decomp = e->mode == HW1F_MODE_DECOMPOSED;
    const size_t smem = cap_smem_bytes(decomp, n, steps[n - 1]);
    HW_TRY(decomp ? set_smem(e, cap_kernel<1>, smem) : set_smem(e, cap_kernel<0>, smem));
    HW_CUDA(e, e->d_cap.ensure(h.size()));
    HW_TRY(upload(e, e->d_cap.p, h.data(), h.size()));
    Launch L;
    HW_TRY(prepare_launch(e, &rng->seed, 1, rng->first_path, rng->n_paths, rng->offset, &L));
    HW_CUDA(e, e->d_partials.ensure((size_t)L.grid_x * nq));
    const ScenDev sc = scen_dev(e, e->p.sigma, e->sig_st, 0);
    const CapletDev* d_caps = reinterpret_cast<const CapletDev*>(e->d_cap.p);
    const float* d_P = reinterpret_cast<const float*>(e->d_cap.p + tab);
    const float sgn = (kind == HW1F_KIND_CAP) ? -1.0f : 1.0f;
    HW_CUDA(e, launch_k(decomp ? cap_kernel<1> : cap_kernel<0>, dim3(L.grid_x, 1), kThreads, smem, e->stream, true, L.g,
                        L.seeds, model_dev(e), sc, d_caps, (int)n, d_P, d_P + nm, sgn, L.lead, e->d_partials.p));
    HW_TRY(check_launch(e, "cap_kernel"));
    HW_TRY(launch_tail(e, L, L.g.n_paths, nq, 0, nullptr, nullptr, 0.f, d_moments, nq, nq, fin));
    rng->offset += (uint64_t)steps[n - 1];
    return HW1F_OK;
}

// P_mkt(T) as interp_mkt evaluates it on the device (IEEE single operations, one fused multiply-add each)
static float host_interp_mkt(const hw1f_engine* e, const float* data, float T)
{
    const int n = e->p.n_mat;
    const float inv = 1.0f / e->spacing;
    const float prod = T * inv;
    const int idx = (prod >= (float)n) ? n : (int)prod;
    if (idx >= n - 1) return data[n - 1];
    const float al = std::fmaf((float)idx, -e->spacing, T) * inv;
    const float om = 1.0f - al;
    return std::fmaf(data[idx], om, al * data[idx + 1]);
}

// double algebra on the pair moments: n_pairs samples of the pair means x = X/2, y = Y/2
static void cap_algebra(const double mom[5], uint64_t n_pairs, double control_mean, hw1f_cap_result* r)
{
    memset(r, 0, sizeof(*r));
    for (int k = 0; k < 5; ++k) r->mom[k] = mom[k];
    const double n = (double)n_pairs;
    const double sx = 0.5 * mom[0], sy = 0.5 * mom[1], sxx = 0.25 * mom[2], syy = 0.25 * mom[3], sxy = 0.25 * mom[4];
    const double mx = sx / n, my = sy / n;
    const double d = n > 1.0 ? n - 1.0 : 1.0;
    double vxx = (sxx - sx * mx) / d, vyy = (syy - sy * my) / d;
    const double cxy = (sxy - sx * my) / d;
    if (vxx < 0.0) vxx = 0.0;
    if (vyy < 0.0) vyy = 0.0;
    const double beta = vyy > 0.0 ? cxy / vyy : 0.0;
    double vcv = vxx - 2.0 * beta * cxy + beta * beta * vyy;
    if (vcv < 0.0) vcv = 0.0;
    r->price_raw = mx;
    r->se_raw = sqrt(vxx / n);
    r->beta = beta;
    r->price_cv = mx - beta * (my - control_mean);
    r->se_cv = sqrt(vcv / n);
    r->corr = (vxx > 0.0 && vyy > 0.0) ? cxy / sqrt(vxx * vyy) : 0.0;
    r->control_mean = control_mean;
}

static void cap_results(const hw1f_engine* e, const double* mom, uint64_t n_pairs, const hw1f_caplet* caps, int32_t n,
                        const float* P_mkt, hw1f_cap_result* out)
{
    double strip_mean = 0.0;
    for (int i = 0; i < n; ++i) {
        const double cm = (double)caps[i].N * (double)host_interp_mkt(e, P_mkt, caps[i].T_pay);
        strip_mean += cm;
        cap_algebra(mom + 5 * i, n_pairs, cm, out + i);
    }
    cap_algebra(mom + 5 * n, n_pairs, strip_mean, out + n);
}

int hw1f_cap_floor_moments(hw1f_engine* e, hw1f_rng* rng, int32_t kind, const hw1f_caplet* caps, int32_t n,
                           const float* P_mkt, const float* f_mkt, double* d_moments)
{
    HW_TRY(require_model(e));
    if (!rng || !caps || !P_mkt || !f_mkt || !d_moments) return HW1F_ERR_INVALID;
    std::vector<int> steps;
    HW_TRY(cap_validate(e, kind, caps, n, steps));
    HW_CUDA(e, cudaSetDevice(e->device));
    Finish fin;
    fin.exchange = true;   // with peers attached (hw1f_comm_attach) the last block all-reduces the vector itself
    return cap_run(e, rng, kind, caps, n, steps, P_mkt, f_mkt, d_moments, fin);
}

int hw1f_cap_floor_finish(hw1f_engine* e, const double* d_moments, uint64_t n_paths_total, const hw1f_caplet* caps,
                          int32_t n, const float* P_mkt, hw1f_cap_result* out)
{
    HW_TRY(require_model(e));
    if (!d_moments || !caps || !P_mkt || !out) return HW1F_ERR_INVALID;
    HW_REQUIRE(e, n_paths_total >= 1 && n_paths_total < (1ull << 40), "n_paths_total outside [1, 2^40)");
    std::vector<int> steps;
    HW_TRY(cap_validate(e, HW1F_KIND_CAP, caps, n, steps));
    HW_CUDA(e, cudaSetDevice(e->device));
    std::vector<double> mom(5 * (size_t)(n + 1));
    HW_TRY(download(e, mom.data(), d_moments, mom.size() * sizeof(double)));
    HW_TRY(require_finite(e, mom.data(), (int)mom.size()));
    cap_results(e, mom.data(), n_paths_total, caps, n, P_mkt, out);
    return HW1F_OK;
}

int hw1f_cap_floor(hw1f_engine* e, hw1f_rng* rng, int32_t kind, const hw1f_caplet* caps, int32_t n, const float* P_mkt,
                   const float* f_mkt, hw1f_cap_result* out, float* sim_ms)
{
    HW_TRY(require_model(e));
    if (!rng || !caps || !P_mkt || !f_mkt || !out) return HW1F_ERR_INVALID;
    std::vector<int> steps;
    HW_TRY(cap_validate(e, kind, caps, n, steps));
    HW_CUDA(e, cudaSetDevice(e->device));
    const size_t nq = 5 * (size_t)(n + 1);
    HW_CUDA(e, e->d_moments.ensure(std::max(4 * (size_t)e->p.n_mat * kMaxRuns, nq)));
    HW_TRY(warm_geometry(e, rng));
    Finish fin;
    fin.host_mom = res_mom(e, 0);   // the result area holds at least 512 doubles
    if (sim_ms) HW_CUDA(e, cudaEventRecord(e->ev0, e->stream));
    HW_TRY(cap_run(e, rng, kind, caps, n, steps, P_mkt, f_mkt, e->d_moments.p, fin));
    if (sim_ms) HW_CUDA(e, cudaEventRecord(e->ev1, e->stream));
    HW_TRY(wait_results(e));
    std::vector<double> mom(res_mom(e, 0), res_mom(e, 0) + nq);
    HW_TRY(require_finite(e, mom.data(), (int)nq));
    cap_results(e, mom.data(), rng->n_paths, caps, n, P_mkt, out);
    if (sim_ms) HW_CUDA(e, cudaEventElapsedTime(sim_ms, e->ev0, e->ev1));
    return HW1F_OK;
}

// ---- European swaptions -------------------------------------------------------------------------
static_assert(kMaxSwaptions == HW1F_MAX_SWAPTIONS && kMaxSwaptionFlows == HW1F_MAX_SWAPTION_FLOWS, "limits of hw1f.h");
static_assert(sizeof(hw1f_swaption) == 32 && sizeof(hw1f_cash_flow) == 8, "ABI structs of hw1f.h");
// every argument checked before any launch; steps[i] = the resolved exercise step of option i, *n_rows = sum of n_flows
static int swaption_validate(hw1f_engine* e, const hw1f_swaption* sw, int32_t n, const hw1f_cash_flow* flows,
                             int32_t n_flows, std::vector<int>& steps, int* n_rows)
{
    HW_REQUIRE(e, n >= 1 && n <= HW1F_MAX_SWAPTIONS, "n_swaptions must be in [1, HW1F_MAX_SWAPTIONS]");
    HW_REQUIRE(e, n_flows >= 1, "n_flows must be >= 1");
    steps.assign(n, 0);
    const double dt = (double)e->dt;
    long rows = 0;
    for (int i = 0; i < n; ++i) {
        const hw1f_swaption& s = sw[i];
        const std::string at = " (swaption " + std::to_string(i) + ")";
        HW_REQUIRE(e, s.kind == HW1F_KIND_PAYER || s.kind == HW1F_KIND_RECEIVER,
                   "kind must be HW1F_KIND_PAYER or HW1F_KIND_RECEIVER" + at);
        HW_REQUIRE(e, std::isfinite(s.T_exercise) && s.T_exercise > 0.0f, "T_exercise must be finite and positive" + at);
        HW_REQUIRE(e, std::isfinite(s.K) && s.K > 0.0f, "K must be finite and positive" + at);
        HW_REQUIRE(e, std::isfinite(s.N) && s.N > 0.0f, "N must be finite and positive" + at);
        HW_REQUIRE(e, s.n_flows >= 1, "n_flows of a swaption must be >= 1" + at);
        HW_REQUIRE(e, s.first_flow >= 0 && (long)s.first_flow + s.n_flows <= n_flows, "flow range outside flows" + at);
        rows += s.n_flows;
        HW_REQUIRE(e, rows <= HW1F_MAX_SWAPTION_FLOWS, "the book's flows exceed HW1F_MAX_SWAPTION_FLOWS" + at);
        float prev = s.T_exercise;
        for (int j = s.first_flow; j < s.first_flow + s.n_flows; ++j) {
            const hw1f_cash_flow& f = flows[j];
            const std::string fat = " (swaption " + std::to_string(i) + ", flow " + std::to_string(j) + ")";
            HW_REQUIRE(e, std::isfinite(f.T) && f.T > prev,
                       "flow dates must be strictly increasing and after T_exercise" + fat);
            HW_REQUIRE(e, std::isfinite(f.c) && f.c > 0.0f, "c must be finite and positive" + fat);
            prev = f.T;
        }
        HW_REQUIRE(e, prev <= e->p.T_final, "the last flow date must not exceed T_final" + at);
        long k = s.n_steps_exercise;
        if (k < 0) {
            k = std::lround((double)s.T_exercise / dt);
            HW_REQUIRE(e, std::fabs((double)s.T_exercise - (double)k * dt) <= 1e-3 * dt,
                       "T_exercise is not on the step grid (|T_exercise - k dt| > 1e-3 dt): pass n_steps_exercise" + at);
        }
        HW_REQUIRE(e, k >= 1 && k <= e->p.n_steps, "exercise step outside [1, n_steps]" + at);
        HW_REQUIRE(e, i == 0 || k >= steps[i - 1], "exercise steps must be non-decreasing along the book" + at);
        steps[i] = (int)k;
    }
    *n_rows = (int)rows;
    return HW1F_OK;
}

// one staged upload of [option table | flow table | P_mkt | f_mkt], the launch and its tail.  The flow table holds each
// option's flows in its own contiguous rows, with its exercise date beside them.
static int swaption_run(hw1f_engine* e, hw1f_rng* rng, const hw1f_swaption* sw, int32_t n, const hw1f_cash_flow* flows,
                        const std::vector<int>& steps, int n_rows, const float* P_mkt, const float* f_mkt,
                        double* d_moments, const Finish& fin)
{
    const int nm = e->p.n_mat, nq = 5 * (n + 1);
    const size_t tab = ((size_t)n * sizeof(SwaptionDev) + 255) & ~(size_t)255;
    const size_t ftab = ((size_t)n_rows * sizeof(SwFlowDev) + 255) & ~(size_t)255;
    std::vector<char> h(tab + ftab + 2 * (size_t)nm * sizeof(float), 0);
    SwaptionDev* sd = reinterpret_cast<SwaptionDev*>(h.data());
    SwFlowDev* fd = reinterpret_cast<SwFlowDev*>(h.data() + tab);
    int row = 0;
    for (int i = 0; i < n; ++i) {
        sd[i].T_e = sw[i].T_exercise;
        sd[i].K = sw[i].K;
        sd[i].N = sw[i].N;
        sd[i].sgn = (sw[i].kind == HW1F_KIND_PAYER) ? -1.0f : 1.0f;
        sd[i].m = (float)e->det_m[0][steps[i]];
        sd[i].Im = (float)e->det_I[0][steps[i]];
        sd[i].step = steps[i];
        sd[i].f0 = row;
        sd[i].nf = sw[i].n_flows;
        for (int j = 0; j < sw[i].n_flows; ++j, ++row) {
            fd[row].T_e = sw[i].T_exercise;
            fd[row].T = flows[sw[i].first_flow + j].T;
            fd[row].c = flows[sw[i].first_flow + j].c;
        }
    }
    memcpy(h.data() + tab + ftab, P_mkt, nm * sizeof(float));
    memcpy(h.data() + tab + ftab + nm * sizeof(float), f_mkt, nm * sizeof(float));
    const int decomp = e->mode == HW1F_MODE_DECOMPOSED;
    const size_t smem = swaption_smem_bytes(decomp, n, n_rows, steps[n - 1]);
    HW_TRY(decomp ? set_smem(e, swaption_kernel<1>, smem) : set_smem(e, swaption_kernel<0>, smem));
    HW_CUDA(e, e->d_cap.ensure(h.size()));
    HW_TRY(upload(e, e->d_cap.p, h.data(), h.size()));
    Launch L;
    HW_TRY(prepare_launch(e, &rng->seed, 1, rng->first_path, rng->n_paths, rng->offset, &L));
    HW_CUDA(e, e->d_partials.ensure((size_t)L.grid_x * nq));
    const ScenDev sc = scen_dev(e, e->p.sigma, e->sig_st, 0);
    const SwaptionDev* d_sw = reinterpret_cast<const SwaptionDev*>(e->d_cap.p);
    const SwFlowDev* d_fl = reinterpret_cast<const SwFlowDev*>(e->d_cap.p + tab);
    const float* d_P = reinterpret_cast<const float*>(e->d_cap.p + tab + ftab);
    HW_CUDA(e, launch_k(decomp ? swaption_kernel<1> : swaption_kernel<0>, dim3(L.grid_x, 1), kThreads, smem, e->stream,
                        true, L.g, L.seeds, model_dev(e), sc, d_sw, (int)n, d_fl, n_rows, d_P, d_P + nm, L.lead,
                        e->d_partials.p));
    HW_TRY(check_launch(e, "swaption_kernel"));
    HW_TRY(launch_tail(e, L, L.g.n_paths, nq, 0, nullptr, nullptr, 0.f, d_moments, nq, nq, fin));
    rng->offset += (uint64_t)steps[n - 1];
    return HW1F_OK;
}

static void swaption_results(const hw1f_engine* e, const double* mom, uint64_t n_pairs, const hw1f_swaption* sw,
                             int32_t n, const hw1f_cash_flow* flows, const float* P_mkt, hw1f_cap_result* out)
{
    double book_mean = 0.0;
    for (int i = 0; i < n; ++i) {
        double annuity = 0.0;
        for (int j = sw[i].first_flow; j < sw[i].first_flow + sw[i].n_flows; ++j)
            annuity += (double)flows[j].c * (double)host_interp_mkt(e, P_mkt, flows[j].T);
        const double cm = (double)sw[i].N * annuity;
        book_mean += cm;
        cap_algebra(mom + 5 * i, n_pairs, cm, out + i);
    }
    cap_algebra(mom + 5 * n, n_pairs, book_mean, out + n);
}

int hw1f_swaptions_moments(hw1f_engine* e, hw1f_rng* rng, const hw1f_swaption* sw, int32_t n,
                           const hw1f_cash_flow* flows, int32_t n_flows, const float* P_mkt, const float* f_mkt,
                           double* d_moments)
{
    HW_TRY(require_model(e));
    if (!rng || !sw || !flows || !P_mkt || !f_mkt || !d_moments) return HW1F_ERR_INVALID;
    std::vector<int> steps;
    int rows = 0;
    HW_TRY(swaption_validate(e, sw, n, flows, n_flows, steps, &rows));
    HW_CUDA(e, cudaSetDevice(e->device));
    Finish fin;
    fin.exchange = true;   // with peers attached (hw1f_comm_attach) the last block all-reduces the vector itself
    return swaption_run(e, rng, sw, n, flows, steps, rows, P_mkt, f_mkt, d_moments, fin);
}

int hw1f_swaptions_finish(hw1f_engine* e, const double* d_moments, uint64_t n_paths_total, const hw1f_swaption* sw,
                          int32_t n, const hw1f_cash_flow* flows, int32_t n_flows, const float* P_mkt,
                          hw1f_cap_result* out)
{
    HW_TRY(require_model(e));
    if (!d_moments || !sw || !flows || !P_mkt || !out) return HW1F_ERR_INVALID;
    HW_REQUIRE(e, n_paths_total >= 1 && n_paths_total < (1ull << 40), "n_paths_total outside [1, 2^40)");
    std::vector<int> steps;
    int rows = 0;
    HW_TRY(swaption_validate(e, sw, n, flows, n_flows, steps, &rows));
    HW_CUDA(e, cudaSetDevice(e->device));
    std::vector<double> mom(5 * (size_t)(n + 1));
    HW_TRY(download(e, mom.data(), d_moments, mom.size() * sizeof(double)));
    HW_TRY(require_finite(e, mom.data(), (int)mom.size()));
    swaption_results(e, mom.data(), n_paths_total, sw, n, flows, P_mkt, out);
    return HW1F_OK;
}

int hw1f_swaptions(hw1f_engine* e, hw1f_rng* rng, const hw1f_swaption* sw, int32_t n, const hw1f_cash_flow* flows,
                   int32_t n_flows, const float* P_mkt, const float* f_mkt, hw1f_cap_result* out, float* sim_ms)
{
    HW_TRY(require_model(e));
    if (!rng || !sw || !flows || !P_mkt || !f_mkt || !out) return HW1F_ERR_INVALID;
    std::vector<int> steps;
    int rows = 0;
    HW_TRY(swaption_validate(e, sw, n, flows, n_flows, steps, &rows));
    HW_CUDA(e, cudaSetDevice(e->device));
    const size_t nq = 5 * (size_t)(n + 1);
    HW_CUDA(e, e->d_moments.ensure(std::max(4 * (size_t)e->p.n_mat * kMaxRuns, nq)));
    HW_TRY(warm_geometry(e, rng));
    Finish fin;
    fin.host_mom = res_mom(e, 0);   // the result area holds at least 512 doubles
    if (sim_ms) HW_CUDA(e, cudaEventRecord(e->ev0, e->stream));
    HW_TRY(swaption_run(e, rng, sw, n, flows, steps, rows, P_mkt, f_mkt, e->d_moments.p, fin));
    if (sim_ms) HW_CUDA(e, cudaEventRecord(e->ev1, e->stream));
    HW_TRY(wait_results(e));
    std::vector<double> mom(res_mom(e, 0), res_mom(e, 0) + nq);
    HW_TRY(require_finite(e, mom.data(), (int)nq));
    swaption_results(e, mom.data(), rng->n_paths, sw, n, flows, P_mkt, out);
    if (sim_ms) HW_CUDA(e, cudaEventElapsedTime(sim_ms, e->ev0, e->ev1));
    return HW1F_OK;
}

// ---- sample paths / introspection ---------------------------------------------------------------
static int run_scalar_kernel(hw1f_engine* e, const hw1f_rng* rng, uint64_t path0, int n_show, float* d_paths,
                             uint32_t* d_state, uint32_t* d_draws, int n_draws, float* d_normals, int n_normals)
{
    Launch L;
    HW_TRY(prepare_launch(e, &rng->seed, 1, rng->first_path + path0, (uint64_t)n_show, rng->offset, &L));
    const ScenDev sc = scen_dev(e, e->p.sigma, e->sig_st, 0);
    HW_CUDA(e, e->d_out.ensure((size_t)e->p.n_steps + 8));
    // plain (non-duplicated) drift table for the scalar kernel
    float* d_drift = e->d_out.p;
    HW_TRY(upload(e, d_drift, e->h_drift.data(), e->p.n_steps * sizeof(float)));
    const int threads = 32, blocks = (n_show + threads - 1) / threads;
    sample_paths_kernel<<<blocks, threads, 0, e->stream>>>(L.g, L.seeds, model_dev(e), sc, n_show, L.lead, d_drift,
                                                           d_paths, d_state, d_draws, n_draws, d_normals, n_normals);
    return check_launch(e, "sample_paths_kernel");
}

int hw1f_sample_paths(hw1f_engine* e, const hw1f_rng* rng, int32_t n_show, float* r_paths)
{
    HW_TRY(require_model(e));
    if (!rng || !r_paths) return HW1F_ERR_INVALID;
    HW_REQUIRE(e, n_show >= 1 && (uint64_t)n_show <= rng->n_paths && n_show <= 65536, "n_show out of range");
    HW_CUDA(e, cudaSetDevice(e->device));
    const size_t n = (size_t)n_show * (e->p.n_steps + 1);
    DevBuf<float> buf;
    HW_CUDA(e, buf.ensure(n));
    int s = run_scalar_kernel(e, rng, 0, n_show, buf.p, nullptr, nullptr, 0, nullptr, 0);
    if (s == HW1F_OK) s = download(e, r_paths, buf.p, n * sizeof(float));
    buf.release();
    return s;
}

int hw1f_debug_rng(hw1f_engine* e, const hw1f_rng* rng, uint64_t path, int32_t n_draws, uint32_t* state6,
                   uint32_t* draws)
{
    HW_TRY(require_model(e));
    if (!rng || !state6) return HW1F_ERR_INVALID;
    HW_REQUIRE(e, path < rng->n_paths && n_draws >= 0 && n_draws <= (1 << 20), "path / n_draws out of range");
    HW_REQUIRE(e, (rng->offset & 1) == 0, "hw1f_debug_rng needs an even normal offset");
    HW_CUDA(e, cudaSetDevice(e->device));
    DevBuf<uint32_t> buf;
    HW_CUDA(e, buf.ensure(6 + (size_t)n_draws));
    int s = run_scalar_kernel(e, rng, path, 1, nullptr, buf.p, n_draws ? buf.p + 6 : nullptr, n_draws, nullptr, 0);
    std::vector<uint32_t> host(6 + (size_t)n_draws);
    if (s == HW1F_OK) s = download(e, host.data(), buf.p, host.size() * sizeof(uint32_t));
    buf.release();
    if (s != HW1F_OK) return s;
    memcpy(state6, host.data(), 6 * sizeof(uint32_t));
    if (draws && n_draws) memcpy(draws, host.data() + 6, (size_t)n_draws * sizeof(uint32_t));
    return HW1F_OK;
}

int hw1f_debug_normals(hw1f_engine* e, const hw1f_rng* rng, uint64_t path, int32_t n, float* out)
{
    HW_TRY(require_model(e));
    if (!rng || !out) return HW1F_ERR_INVALID;
    HW_REQUIRE(e, path < rng->n_paths && n >= 1 && n <= (1 << 20), "path / n out of range");
    HW_CUDA(e, cudaSetDevice(e->device));
    DevBuf<float> buf;
    HW_CUDA(e, buf.ensure((size_t)n));
    int s = run_scalar_kernel(e, rng, path, 1, nullptr, nullptr, nullptr, 0, buf.p, n);
    if (s == HW1F_OK) s = download(e, out, buf.p, (size_t)n * sizeof(float));
    buf.release();
    return s;
}

int hw1f_reduction_bench(hw1f_engine* e, hw1f_rng* rng, int32_t method, float S1, float S2, float K,
                         const float* P_mkt, const float* f_mkt, int32_t n_steps_S1, int32_t n_warmup, int32_t n_runs,
                         float* avg_ms, float* price)
{
    HW_TRY(require_model(e));
    if (!rng || !P_mkt || !f_mkt || !avg_ms || !price) return HW1F_ERR_INVALID;
    HW_REQUIRE(e, method >= 0 && method <= 3 && n_runs >= 1 && n_warmup >= 0, "method in [0,3], n_runs >= 1");
    HW_CUDA(e, cudaSetDevice(e->device));
    int32_t n = 0;
    HW_TRY(resolve_steps(e, S1, n_steps_S1, &n));
    const ScenDev sc = scen_dev(e, e->p.sigma, e->sig_st, 0);
    HW_TRY(launch_plan_job(e, plan_job_host(e, &sc, 1, S1, S2, P_mkt, f_mkt)));
    HW_CUDA(e, e->d_moments.ensure(4 * (size_t)e->p.n_mat * kMaxRuns));
    HW_CUDA(e, e->d_out.ensure(64));
    float* d_sum = e->d_out.p;
    const size_t smem = (size_t)kWinWords * 4 + (size_t)((n + 1) / 2 + 1) * sizeof(float4);
    HW_TRY(set_smem(e, zbc_sum_kernel<0>, smem));
    HW_TRY(set_smem(e, zbc_sum_kernel<1>, smem));
    HW_TRY(set_smem(e, zbc_sum_kernel<2>, smem));
    HW_TRY(set_smem(e, zbc_sum_kernel<3>, smem));
    double total_ms = 0.0;
    // benchmark_kernel(), src/benchmark_reductions.cu:34-54: warm-ups then timed launches, each launch
    // continues the streams (states are written back there; the handle offset advances here)
    for (int it = 0; it < n_warmup + n_runs; ++it) {
        Launch L;
        HW_CUDA(e, cudaMemsetAsync(d_sum, 0, sizeof(float), e->stream));
        HW_CUDA(e, cudaEventRecord(e->ev0, e->stream));
        HW_TRY(prepare_launch(e, &rng->seed, 1, rng->first_path, rng->n_paths, rng->offset, &L));
        HW_CUDA(e, e->d_partials.ensure((size_t)L.grid_x));
        const ModelDev md = model_dev(e);
        switch (method) {
            case 0: zbc_sum_kernel<0><<<L.grid_x, kThreads, smem, e->stream>>>(L.g, L.seeds, md, sc, e->d_plans.p, n, L.lead, K, d_sum, e->d_partials.p); break;
            case 1: zbc_sum_kernel<1><<<L.grid_x, kThreads, smem, e->stream>>>(L.g, L.seeds, md, sc, e->d_plans.p, n, L.lead, K, d_sum, e->d_partials.p); break;
            case 2: zbc_sum_kernel<2><<<L.grid_x, kThreads, smem, e->stream>>>(L.g, L.seeds, md, sc, e->d_plans.p, n, L.lead, K, d_sum, e->d_partials.p); break;
            default: zbc_sum_kernel<3><<<L.grid_x, kThreads, smem, e->stream>>>(L.g, L.seeds, md, sc, e->d_plans.p, n, L.lead, K, d_sum, e->d_partials.p); break;
        }
        HW_TRY(check_launch(e, "zbc_sum_kernel"));
        if (method == 3) HW_TRY(reduce_to(e, 1, L.grid_x, 1, e->d_moments.p));
        HW_CUDA(e, cudaEventRecord(e->ev1, e->stream));
        HW_CUDA(e, cudaEventSynchronize(e->ev1));
        rng->offset += (uint64_t)n;
        if (it >= n_warmup) {
            float ms = 0.f;
            HW_CUDA(e, cudaEventElapsedTime(&ms, e->ev0, e->ev1));
            total_ms += ms;
        }
    }
    *avg_ms = (float)(total_ms / n_runs);
    if (method == 3) {
        double s = 0.0;
        HW_TRY(download(e, &s, e->d_moments.p, sizeof(double)));
        *price = (float)s / (2.0f * (float)rng->n_paths);       // h_sum / (2.0f * N_PATHS), src/bench:62
    } else {
        float s = 0.f;
        HW_TRY(download(e, &s, d_sum, sizeof(float)));
        *price = s / (2.0f * (float)rng->n_paths);
    }
    return HW1F_OK;
}

// state after curand_init(seed, path, 2*floor(normal_offset/2)) computed on the HOST by the
// engine's own jump algebra (no GPU needed): state6 = {d, v0..v4}
int hw1f_host_rng_state(uint64_t seed, uint64_t path, uint64_t normal_offset, uint32_t* state6)
{
    if (!state6) return HW1F_ERR_INVALID;
    const JumpTables& jt = jump_tables();
    BitVec v;
    const uint32_t d0 = seed_scramble(seed, v);
    uint64_t sub = path;
    for (int k = 0; sub != 0 && k < kNumPow; ++k, sub >>= 1)
        if (sub & 1) v = jt.seq_pow2[k].apply(v);
    if (sub != 0) return HW1F_ERR_UNSUPPORTED;
    const uint64_t draws = 2 * (normal_offset / 2);
    uint64_t off = draws;
    for (int k = 0; off != 0 && k < kNumPow; ++k, off >>= 1)
        if (off & 1) v = jt.step_pow2[k].apply(v);
    if (off != 0) return HW1F_ERR_UNSUPPORTED;
    state6[0] = d0 + kWeyl * (uint32_t)draws;
    for (int w = 0; w < 5; ++w) state6[1 + w] = v[w];
    return HW1F_OK;
}

int hw1f_pipe_probe(hw1f_engine* e, int32_t which, int32_t iters, float* ms, double* thread_instr)
{
    if (!e || !ms || !thread_instr) return HW1F_ERR_INVALID;
    HW_REQUIRE(e, which >= 0 && which <= 13 && iters >= 1, "which in [0,13], iters >= 1");
    HW_CUDA(e, cudaSetDevice(e->device));
    HW_CUDA(e, e->d_out.ensure(64));
    const int blocks = e->sm_count * 8, threads = 256;
    for (int rep = 0; rep < 2; ++rep) {   // first pass warms the instruction cache and clocks
        HW_CUDA(e, cudaEventRecord(e->ev0, e->stream));
        switch (which) {
            case 0: probe_kernel<0><<<blocks, threads, 0, e->stream>>>(iters, 1.0f, 12345u, e->d_out.p); break;
            case 1: probe_kernel<1><<<blocks, threads, 0, e->stream>>>(iters, 1.0f, 12345u, e->d_out.p); break;
            case 2: probe_kernel<2><<<blocks, threads, 0, e->stream>>>(iters, 1.0f, 12345u, e->d_out.p); break;
            case 3: probe_kernel<3><<<blocks, threads, 0, e->stream>>>(iters, 1.0f, 12345u, e->d_out.p); break;
            case 4: probe_kernel<4><<<blocks, threads, 0, e->stream>>>(iters, 1.0f, 12345u, e->d_out.p); break;
            case 5: probe_kernel<5><<<blocks, threads, 0, e->stream>>>(iters, 1.0f, 12345u, e->d_out.p); break;
            case 6: probe_kernel<6><<<blocks, threads, 0, e->stream>>>(iters, 1.0f, 12345u, e->d_out.p); break;
            case 7: probe_kernel<7><<<blocks, threads, 0, e->stream>>>(iters, 1.0f, 12345u, e->d_out.p); break;
            case 8: probe_kernel<8><<<blocks, threads, 0, e->stream>>>(iters, 1.0f, 12345u, e->d_out.p); break;
            case 9: probe_kernel<9><<<blocks, threads, 0, e->stream>>>(iters, 1.0f, 12345u, e->d_out.p); break;
            case 10: probe_kernel<10><<<blocks, threads, 0, e->stream>>>(iters, 1.0f, 12345u, e->d_out.p); break;
            case 11: probe_kernel<11><<<blocks, threads, 0, e->stream>>>(iters, 1.0f, 12345u, e->d_out.p); break;
            case 12: probe_kernel<12><<<blocks, threads, 0, e->stream>>>(iters, 1.0f, 12345u, e->d_out.p); break;
            default: probe_kernel<13><<<blocks, threads, 0, e->stream>>>(iters, 1.0f, 12345u, e->d_out.p); break;
        }
        HW_TRY(check_launch(e, "probe_kernel"));
        HW_CUDA(e, cudaEventRecord(e->ev1, e->stream));
        HW_CUDA(e, cudaEventSynchronize(e->ev1));
    }
    HW_CUDA(e, cudaEventElapsedTime(ms, e->ev0, e->ev1));
    // probed instructions per thread (for 4/5: the conversion or the MUFU count; the feeder ops are extra;
    // 10-13: MUFU only -- the other instructions of 13 are the load the MUFU rate is measured under)
    const double per_thread = (which == 6) ? (double)iters * kProbeUnroll * 29.0
                                           : (double)iters * kProbeUnroll * kProbeChains;
    *thread_instr = per_thread * (double)blocks * threads;
    return HW1F_OK;
}

// engine side of hw1f_comm_attach (hw1f_comm.cu); not part of the public header
int hw1f_engine_attach_comm_internal(hw1f_engine* e, const void* comm_dev, unsigned* epoch, int on)
{
    if (!e || (on && (!comm_dev || !epoch))) return HW1F_ERR_INVALID;
    HW_CUDA(e, cudaSetDevice(e->device));
    HW_CUDA(e, cudaStreamSynchronize(e->stream));
    e->comm_on = on != 0;
    if (on) {
        e->comm = *static_cast<const CommDev*>(comm_dev);
        e->comm_epoch = epoch;
    } else {
        e->comm = CommDev{};
        e->comm_epoch = nullptr;
    }
    return HW1F_OK;
}

int hw1f_launch_count(const hw1f_engine* e, uint64_t* n)
{
    if (!e || !n) return HW1F_ERR_INVALID;
    *n = e->launches;
    for (auto t : e->twin) if (t) *n += t->launches;
    return HW1F_OK;
}

}  // extern "C"
