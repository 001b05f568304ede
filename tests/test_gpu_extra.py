"""GPU tests of the wider surface: the fused pass, the reduction benchmark, and the four drop-in
drivers run end to end next to the reference's own binaries (seeds pinned on both sides)."""
import json
import os
import subprocess

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
N = 1 << 14
SEED = 4242
# the drivers' time(NULL) seed, pinned: the seed of the stored reference run tests/golden/ref_b200_seed20251018.json
DRIVER_SEED = 20251018


@pytest.fixture(scope="module")
def curve(engine, hw):
    return engine.bond_curve(hw.Rng(SEED, N))


def test_fused_equals_separate_passes(engine, hw, curve):
    """one launch, one set of normals == the three separate estimators on the same window"""
    import ctypes as C
    nm = engine.n_mat
    fused = torch.zeros(2 * nm + 8, dtype=torch.float64, device="cuda")
    sep_c = torch.zeros(2 * nm, dtype=torch.float64, device="cuda")
    sep_z = torch.zeros(5, dtype=torch.float64, device="cuda")
    sep_v = torch.zeros(2, dtype=torch.float64, device="cuda")
    torch.cuda.synchronize()
    P, f = np.ascontiguousarray(curve["P"]), np.ascontiguousarray(curve["f"])
    lib = hw._ffi.load()
    rng = hw.Rng(SEED, N)
    st = lib.hw1f_fused_moments(engine._h, rng._h, 5.0, 10.0, engine.K_DEFAULT, P.ctypes.data_as(C.c_void_p),
                                f.ctypes.data_as(C.c_void_p), 500, C.c_void_p(fused.data_ptr()))
    assert st == 0, lib.hw1f_last_error(engine._h)
    assert rng.tell() == 1000
    engine.bond_curve_moments(hw.Rng(SEED, N), sep_c.data_ptr())
    engine.zbc_cv_moments(hw.Rng(SEED, N), P, f, sep_z.data_ptr(), n_steps_S1=500)
    engine.vega_pathwise_moments(hw.Rng(SEED, N), P, f, sep_v.data_ptr(), n_steps_S1=500)
    engine.synchronize()
    fused, sep_c, sep_z, sep_v = (t.cpu().numpy() for t in (fused, sep_c, sep_z, sep_v))
    assert np.allclose(fused[1:nm], sep_c[1:nm], rtol=1e-12) and np.allclose(fused[nm + 1:2 * nm], sep_c[nm + 1:], rtol=1e-10)
    assert np.allclose(fused[2 * nm:2 * nm + 5], sep_z, rtol=1e-13)
    # +G twin == the non-antithetic pathwise kernel (different template instantiations may round a
    # handful of per-path values differently by one ulp: compare to 1e-7, not bit for bit)
    assert fused[2 * nm + 7] == pytest.approx(sep_v[0], rel=1e-7)
    both = fused[2 * nm + 5] / (2 * N)
    assert abs(both - sep_v[0] / N) < 0.02                              # antithetic twin: same estimand


def test_reduction_bench_methods(engine, hw, curve, oracle):
    """hw1f_reduction_bench (perf_benchmark.cuh:19-197, src/benchmark_reductions.cu:17-72) against the ORACLE: every
    launch continues the streams, so launch j of the shared handle sees normals [500 j, 500 j + 500)"""
    n, steps = 1 << 16, 500
    P, f = curve["P"], curve["f"]
    rng = hw.Rng(SEED, n)
    launches_per_method = 3                                   # 1 warm-up + 2 timed; the price is the LAST launch's
    for method in range(4):
        r = engine.reduction_bench(rng, method, P, f, n_steps_S1=steps, n_warmup=1, n_runs=2)
        assert r["avg_ms"] > 0
        last = method * launches_per_method + launches_per_method - 1
        mom = oracle.zbc_moments(SEED, n, P, f, n_steps_S1=steps, offset=last * steps)
        want = mom[0] / (2.0 * n)
        if method == 3:      # deterministic two-level tree in double: the oracle's sum to float32 rounding
            assert r["price"] == pytest.approx(want, rel=3e-6), (method, r["price"], want)
        else:                # float32 atomics (order-dependent rounding, like the reference's): measured <= 2e-5
            assert r["price"] == pytest.approx(want, rel=1e-4), (method, r["price"], want)
    assert rng.tell() == 4 * launches_per_method * steps
    # the tree on the window of zbc_cv reproduces its raw price
    ref = engine.zbc_cv(hw.Rng(SEED, n), P, f, n_steps_S1=steps)
    one = engine.reduction_bench(hw.Rng(SEED, n), 3, P, f, n_steps_S1=steps, n_warmup=0, n_runs=1)
    assert one["price"] == pytest.approx(ref["price_raw"], rel=1e-6)


# ---------------------------------------------------------------- drivers, end to end
def _run(cmd, cwd, stdin="", env=None):
    e = dict(os.environ)
    e.update(env or {})
    return subprocess.run(cmd, cwd=cwd, input=stdin, text=True, capture_output=True, env=e, timeout=900)


@pytest.fixture(scope="module")
def driver_runs(tmp_path_factory):
    bins = os.path.join(ROOT, "bin")
    if not all(os.path.exists(os.path.join(bins, b)) for b in ("q1", "q2", "q3", "benchmark")):
        pytest.skip("bin/ drivers not built (make all benchmark)")
    mine = tmp_path_factory.mktemp("mine")
    os.makedirs(mine / "data")
    env = {"HW_SEED": str(DRIVER_SEED), "HW_DEVICE": "0"}
    logs = {}
    logs["q1"] = _run([os.path.join(bins, "q1")], mine, env=env)
    logs["q2"] = _run([os.path.join(bins, "q2")], mine, stdin="y\n", env=env)
    logs["q3"] = _run([os.path.join(bins, "q3")], mine, stdin="n\ny\n", env=env)
    logs["benchmark"] = _run([os.path.join(bins, "benchmark")], mine, env=env)
    ref = None
    refbin = os.path.join(ROOT, "oracle", "_ref")
    if os.path.exists(os.path.join(refbin, "q1")):
        ref = tmp_path_factory.mktemp("ref")
        os.makedirs(ref / "data")
        renv = {"LD_PRELOAD": os.path.join(refbin, "libfaketime.so"), "HW1F_FAKE_TIME": str(DRIVER_SEED)}
        for q, stdin in (("q1", ""), ("q2", "y\n"), ("q3", "n\ny\n"), ("benchmark", "")):
            logs["ref_" + q] = _run([os.path.join(refbin, q)], ref, stdin=stdin, env=renv)
    return mine, ref, logs


def test_drivers_write_the_frozen_schema(driver_runs):
    mine, ref, logs = driver_runs
    for q in ("q1", "q2", "q3", "benchmark"):
        assert logs[q].returncode == 0, logs[q].stdout[-2000:] + logs[q].stderr[-2000:]
    data = mine / "data"
    expected = ["P.bin", "f.bin", "r_paths.bin", "q1_results.json", "P_curve.csv", "f_curve.csv", "summary.txt",
                "q2a_results.json", "theta_comparison.csv", "zbc_bootstrap_optimal.csv", "zbc_statistics_optimal.txt",
                "q3_results.json", "vega_bootstrap.csv", "vega_statistics.txt", "benchmark_reductions.json"]
    for name in expected:
        assert (data / name).exists(), name
    assert np.fromfile(data / "P.bin", np.float32).shape == (101,)
    assert np.fromfile(data / "r_paths.bin", np.float32).shape == (32 * 1001,)
    q1 = json.load(open(data / "q1_results.json"))
    assert set(q1) == {"task", "timestamp", "parameters", "P", "f", "performance", "validation"}
    assert set(q1["parameters"]) == {"N_PATHS", "N_STEPS", "N_MAT", "T_FINAL", "a", "sigma", "r0"}
    assert set(q1["performance"]) == {"simulation_time_ms", "throughput_Mpaths_per_sec"}
    assert set(q1["validation"]) == {"P_0_0", "P_0_10", "f_0_0"}
    q2a = json.load(open(data / "q2a_results.json"))
    assert set(q2a["error_metrics"]) == {"max_error", "success"} and q2a["error_metrics"]["success"] is True
    q3 = json.load(open(data / "q3_results.json"))
    assert set(q3["results"]) == {"sensitivity_mc", "sensitivity_fd", "abs_diff"}
    br = json.load(open(data / "benchmark_reductions.json"))
    assert len(br["results"]) == 4 and set(br["results"][0]) == {"method", "time_ms", "throughput_Mpaths_per_sec", "price"}
    assert open(data / "theta_comparison.csv").readline().strip() == "T,theta_original,theta_recovered"
    assert open(data / "zbc_bootstrap_optimal.csv").readline().strip() == "run,price_adjusted,price_raw,beta_optimal,correlation"
    assert open(data / "vega_bootstrap.csv").readline().strip() == "run,vega"
    assert len(open(data / "vega_bootstrap.csv").readlines()) == 21


def test_drivers_match_reference_fixture(driver_runs, golden_dir):
    """our q1 / q2 / q3 drivers against the stored run of the unmodified reference kernels with the same seed
    (oracle/ref/ref_harness.cu `parity`: the reference's Q1 main, sample paths, theta recovery and Q3 main); the bounds
    are those of the live comparison below"""
    mine, _, logs = driver_runs
    for q in ("q1", "q2", "q3"):
        assert logs[q].returncode == 0, logs[q].stdout[-1500:]
    with open(os.path.join(golden_dir, "ref_b200_seed20251018.json")) as fh:
        ref = json.load(fh)
    assert ref["seed"] == DRIVER_SEED
    Pm, Pr = np.fromfile(mine / "data" / "P.bin", np.float32), np.array(ref["P"], np.float32)
    fm, fr = np.fromfile(mine / "data" / "f.bin", np.float32), np.array(ref["f"], np.float32)
    assert np.abs(Pm / Pr - 1).max() < 3e-5 and np.abs(Pm[20:] / Pr[20:] - 1).max() < 1e-5
    assert np.abs(fm - fr).max() < 3e-4
    rm = np.fromfile(mine / "data" / "r_paths.bin", np.float32).reshape(32, -1)
    assert np.abs(rm[0] - np.array(ref["r_path0"], np.float32)).max() < 2e-6
    assert np.abs(rm[31] - np.array(ref["r_path31"], np.float32)).max() < 2e-6
    tm = np.loadtxt(mine / "data" / "theta_comparison.csv", delimiter=",", skiprows=1)
    assert np.abs(tm[:, 1] - np.array(ref["theta_orig"], np.float32)).max() < 1e-8    # analytic theta, "%.8f" in the CSV
    th = np.array(ref["theta_rec"], np.float32)
    assert np.abs(tm[10:, 2] - th[10:]).max() < 10 * np.abs(fm[9:] - fr[9:]).max() + 1e-6
    q3m = json.load(open(mine / "data" / "q3_results.json"))["results"]
    assert q3m["sensitivity_mc"] == pytest.approx(ref["vega_pathwise"], rel=2e-4)
    assert q3m["sensitivity_fd"] == pytest.approx(ref["vega_fd"], abs=1e-3)


def test_drivers_match_reference_binaries(driver_runs):
    """the unmodified reference drivers (sm_100 rebuild, time() pinned by LD_PRELOAD) next to ours"""
    mine, ref, logs = driver_runs
    if ref is None:
        pytest.skip("oracle/_ref binaries not built")
    for q in ("ref_q1", "ref_q2", "ref_q3"):
        assert logs[q].returncode == 0, logs[q].stdout[-1500:]
    Pm, Pr = (np.fromfile(d / "data" / "P.bin", np.float32) for d in (mine, ref))
    fm, fr = (np.fromfile(d / "data" / "f.bin", np.float32) for d in (mine, ref))
    assert np.abs(Pm / Pr - 1).max() < 3e-5 and np.abs(Pm[20:] / Pr[20:] - 1).max() < 1e-5
    assert np.abs(fm - fr).max() < 3e-4
    rm, rr = (np.fromfile(d / "data" / "r_paths.bin", np.float32) for d in (mine, ref))
    assert np.abs(rm - rr).max() < 2e-6                      # same 32 trajectories, draw window 1000..1999
    # same schema on both sides
    for name in ("q1_results.json", "q2a_results.json", "q3_results.json"):
        a, b = json.load(open(mine / "data" / name)), json.load(open(ref / "data" / name))
        assert set(a) == set(b), name
    q3m, q3r = (json.load(open(d / "data" / "q3_results.json"))["results"] for d in (mine, ref))
    # both drivers consumed P.bin/f.bin of their own q1; vega agrees to the curve difference
    assert q3m["sensitivity_mc"] == pytest.approx(q3r["sensitivity_mc"], rel=2e-4)
    assert q3m["sensitivity_fd"] == pytest.approx(q3r["sensitivity_fd"], abs=1e-3)
    vm = np.loadtxt(mine / "data" / "vega_bootstrap.csv", delimiter=",", skiprows=1)[:, 1]
    vr = np.loadtxt(ref / "data" / "vega_bootstrap.csv", delimiter=",", skiprows=1)[:, 1]
    assert np.abs(vm / vr - 1).max() < 2e-4                  # 20 seeds, one launch vs 20x(malloc+init+kernel)
    zm = np.loadtxt(mine / "data" / "zbc_bootstrap_optimal.csv", delimiter=",", skiprows=1)
    zr = np.loadtxt(ref / "data" / "zbc_bootstrap_optimal.csv", delimiter=",", skiprows=1)
    assert np.abs(zm[:, 1] / zr[:, 1] - 1).max() < 1e-4      # CV-adjusted prices
    assert np.abs(zm[:, 2] / zr[:, 2] - 1).max() < 1e-4      # raw prices
    # theta recovered from each driver's own forward curve (recover_theta, src/2:14-35): d theta ~ 10 x d f
    tm = np.loadtxt(mine / "data" / "theta_comparison.csv", delimiter=",", skiprows=1)
    tr = np.loadtxt(ref / "data" / "theta_comparison.csv", delimiter=",", skiprows=1)
    assert (tm[:, 0] == tr[:, 0]).all() and np.abs(tm[:, 1] - tr[:, 1]).max() == 0     # T grid, analytic theta
    assert np.abs(tm[10:, 2] - tr[10:, 2]).max() < 10 * np.abs(fm[9:] - fr[9:]).max() + 1e-6
    # the reduction benchmark (src/benchmark_reductions.cu:74-212): same seed, every launch continues the streams, so
    # method k of both drivers prices the same window with the same strategy; float32 atomics on both sides
    assert logs["ref_benchmark"].returncode == 0, logs["ref_benchmark"].stdout[-1500:]
    bm = json.load(open(mine / "data" / "benchmark_reductions.json"))["results"]
    br = json.load(open(ref / "data" / "benchmark_reductions.json"))["results"]
    assert len(br) == 3 and [r["method"] for r in br] == [r["method"] for r in bm[:3]]
    for a, b in zip(bm[:3], br):
        assert a["price"] == pytest.approx(b["price"], rel=1e-4), (a, b)
    # the fourth method (deterministic tree, no reference counterpart) prices the next window: same estimand
    se = 0.045 / np.sqrt(2.0 * (1 << 20))                      # sd of the discounted payoff ~ 0.045
    assert abs(bm[3]["price"] - np.mean([r["price"] for r in br])) < 6 * se


def test_fused_with_fd_bumps_one_launch(engine, hw, curve):
    """hw1f_fused: curve + ZBC/CV + antithetic pathwise vega + CRN FD bumps from ONE launch equal the
    separate entry points evaluated on the same draw window"""
    before = engine.launch_count
    got = engine.fused(hw.Rng(SEED, N), curve["P"], curve["f"], eps=0.001, n_steps_S1=500)
    sim_launches = engine.launch_count - before
    assert sim_launches <= 8                              # plans x2, prep, ONE simulation kernel, reduce, un-centre, epilogue
    sep_curve = engine.bond_curve(hw.Rng(SEED, N))
    assert (got["P"] == sep_curve["P"]).all() and np.abs(got["f"] - sep_curve["f"]).max() == 0
    z = engine.zbc_cv(hw.Rng(SEED, N), curve["P"], curve["f"], n_steps_S1=500)
    assert got["zbc"]["price_cv"] == z["price_cv"] and got["zbc"]["beta"] == z["beta"]
    fd = engine.vega_fd(hw.Rng(SEED, N), curve["P"], curve["f"], eps=0.001, n_steps_S1=500)   # same window [0,500)
    assert got["vega"]["price_minus"] == fd["price_minus"] and got["vega"]["price_plus"] == fd["price_plus"]
    assert got["vega"]["vega_fd"] == fd["vega_fd"]
    pw = engine.vega_pathwise(hw.Rng(SEED, N), curve["P"], curve["f"], n_steps_S1=500)
    assert abs(got["vega"]["vega_pathwise_f64"] - pw["vega_pathwise_f64"]) < 4 * pw["vega_pathwise_se"]
    assert 0 < got["vega"]["vega_pathwise_se"] < pw["vega_pathwise_se"]      # antithetic twins: smaller error


def test_fused_shards_allreduce_finish(engine, hw, curve):
    """the scaling-run shape on one GPU: two disjoint subsequence shards -> hw1f_fused_fd_moments each -> sum of
    the moment vectors (what the all-reduce does) -> hw1f_fused_finish == hw1f_fused over the whole range"""
    import torch
    nm = engine.n_mat
    whole = engine.fused(hw.Rng(SEED, N), curve["P"], curve["f"], eps=0.001, n_steps_S1=500)
    acc = torch.zeros(2 * nm + 18, dtype=torch.float64, device="cuda")
    part = torch.zeros_like(acc)
    torch.cuda.synchronize()
    cut = 5555                                             # ragged split: neither shard is chunk aligned
    for first, cnt in ((0, cut), (cut, N - cut)):
        engine.fused_moments(hw.Rng(SEED, cnt, first_path=first), curve["P"], curve["f"], part.data_ptr(), eps=0.001,
                             n_steps_S1=500)
        engine.synchronize()
        acc += part
    torch.cuda.synchronize()
    got = engine.fused_finish(acc.data_ptr(), N, float(curve["P"][-1]), eps=0.001, n_steps_S1=500)
    assert np.abs(got["P"] / whole["P"] - 1).max() < 2e-7 and np.abs(got["f"] - whole["f"]).max() < 2e-6
    assert np.allclose(got["zbc"]["mom"], whole["zbc"]["mom"], rtol=1e-12)
    assert got["zbc"]["price_cv"] == pytest.approx(whole["zbc"]["price_cv"], rel=1e-6)
    assert got["vega"]["vega_pathwise_f64"] == pytest.approx(whole["vega"]["vega_pathwise_f64"], rel=1e-12)
    assert got["vega"]["vega_fd"] == pytest.approx(whole["vega"]["vega_fd"], rel=1e-4)


def test_finish_beyond_int_range(engine, hw, curve):
    """2*n_paths >= 2^31 (the 2^30-subsequence scaling run) is outside the reference's `int N_total`; the finish
    calls must keep working there.  Moments of a 2^14 run scaled by 2^18 stand in for a 2^32-subsequence run:
    every mean is unchanged, standard errors shrink by sqrt(2^18) = 512."""
    import torch
    SCALE = 1 << 18
    nm = engine.n_mat
    mom = torch.zeros(2 * nm + 18, dtype=torch.float64, device="cuda")
    torch.cuda.synchronize()
    engine.fused_moments(hw.Rng(SEED, N), curve["P"], curve["f"], mom.data_ptr(), eps=0.001, n_steps_S1=500)
    engine.synchronize()
    small = engine.fused_finish(mom.data_ptr(), N, float(curve["P"][-1]), eps=0.001, n_steps_S1=500)
    big_mom = mom * float(SCALE)
    torch.cuda.synchronize()
    big = engine.fused_finish(big_mom.data_ptr(), N * SCALE, float(curve["P"][-1]), eps=0.001, n_steps_S1=500)
    assert big["zbc"]["n_total"] == 2 * N * SCALE and big["zbc"]["n_total"] >= 1 << 31
    assert np.abs(big["P"] / small["P"] - 1).max() < 2e-7 and np.abs(big["f"] - small["f"]).max() < 2e-6
    assert big["zbc"]["price_cv"] == pytest.approx(small["zbc"]["price_cv"], rel=1e-6)
    assert big["zbc"]["beta"] == pytest.approx(small["zbc"]["beta"], rel=1e-5)
    assert big["vega"]["vega_pathwise_f64"] == pytest.approx(small["vega"]["vega_pathwise_f64"], rel=1e-12)
    assert big["vega"]["vega_pathwise_se"] == pytest.approx(small["vega"]["vega_pathwise_se"] / SCALE ** 0.5, rel=1e-3)
    assert big["P_se"][50] == pytest.approx(small["P_se"][50] / SCALE ** 0.5, rel=1e-3)
    z = engine.zbc_cv_finish(big_mom.data_ptr() + 8 * 2 * nm, N * SCALE, float(curve["P"][-1]))
    assert z["price_cv"] == big["zbc"]["price_cv"]


@pytest.mark.parametrize("call", ["zbc_cv", "vega_pathwise", "vega_fd", "vega_fd_recalibrated", "vega", "fused",
                                  "zbc_cv_batch", "vega_pathwise_batch", "sample_paths", "theta"])
def test_every_entry_point_as_first_call_of_a_fresh_engine(engine, hw, curve, call):
    """lazily built state (jump tables, window tables, bumped-sigma arena, scratch) must not depend on what ran
    before: each entry point, called FIRST on a new engine with a ragged path count, reproduces the long-lived
    session engine bit for bit"""
    n = (1 << 12) + 77
    P, f = curve["P"], curve["f"]

    def run(e):
        if call == "zbc_cv":
            return e.zbc_cv(hw.Rng(SEED, n), P, f, n_steps_S1=500)["mom"]
        if call == "vega_pathwise":
            return [e.vega_pathwise(hw.Rng(SEED, n), P, f, n_steps_S1=500)["vega_pathwise_f64"]]
        if call == "vega_fd":
            r = e.vega_fd(hw.Rng(SEED, n), P, f, n_steps_S1=500)
            return [r["price_minus"], r["price_plus"]]
        if call == "vega_fd_recalibrated":
            r = e.vega_fd_recalibrated(hw.Rng(SEED, n), n_steps_S1=500)
            return [r["price_minus_recal"], r["price_plus_recal"]]
        if call == "vega":
            r = e.vega(hw.Rng(SEED, n), P, f, n_steps_S1=500)
            return [r["vega_pathwise_f64"], r["price_minus"], r["price_plus"], r["price_minus_recal"], r["price_plus_recal"]]
        if call == "fused":
            r = e.fused(hw.Rng(SEED, n), P, f, n_steps_S1=500)
            return list(r["P"]) + r["zbc"]["mom"] + [r["vega"]["vega_pathwise_f64"], r["vega"]["price_minus"]]
        if call == "zbc_cv_batch":
            res, _ = e.zbc_cv_batch([SEED, SEED + 1, SEED + 2], n, P, f, n_steps_S1=500)
            return [x for r in res for x in r["mom"]]
        if call == "vega_pathwise_batch":
            v, _ = e.vega_pathwise_batch([SEED, SEED + 1], n, P, f, n_steps_S1=500)
            return list(v)
        if call == "sample_paths":
            return list(e.sample_paths(hw.Rng(SEED, n), 4).ravel())
        return list(e.theta_calibrate(f)["theta_rec"])

    fresh = hw.Engine(device=0)
    fresh.set_mode(engine.mode)
    try:
        first = run(fresh)
    finally:
        fresh.close()
    assert first == run(engine)


def test_changing_path_ranges_on_one_engine(engine, hw, curve):
    """window tables, the per-launch jump table and the scratch buffers are sized per path range: walking through
    different ranges (sizes, first paths) on ONE engine gives what a fresh engine gives for each of them"""
    P, f = curve["P"], curve["f"]
    ranges = [(1 << 14, 0), ((1 << 12) + 77, 0), (1 << 16, 3), (900, (1 << 33) + 5), (1 << 14, 0), (1 << 18, 1 << 20)]
    for n, first in ranges:
        z = engine.zbc_cv(hw.Rng(SEED, n, first_path=first), P, f, n_steps_S1=500)["mom"]
        c = engine.bond_curve(hw.Rng(SEED, n, first_path=first))["P"]
        fresh = hw.Engine(device=0)
        fresh.set_mode(engine.mode)
        try:
            assert z == fresh.zbc_cv(hw.Rng(SEED, n, first_path=first), P, f, n_steps_S1=500)["mom"], (n, first)
            assert (c == fresh.bond_curve(hw.Rng(SEED, n, first_path=first))["P"]).all(), (n, first)
        finally:
            fresh.close()


def test_two_engines_in_two_threads(engine, hw, curve):
    """include/hw1f.h: an engine is not thread-safe, engines share nothing but the GPU -- two host threads, one
    engine each, interleave freely (ctypes releases the GIL inside every call)"""
    import threading
    n = (1 << 14) + 5
    want = {s: engine.zbc_cv(hw.Rng(s, n), curve["P"], curve["f"], n_steps_S1=500)["mom"] for s in range(100, 108)}
    wantc = {s: engine.bond_curve(hw.Rng(s, n))["P"] for s in range(100, 108)}
    errors = []

    def worker(seeds):
        try:
            e = hw.Engine(device=0)
            e.set_mode(engine.mode)
            for _ in range(3):
                for s in seeds:
                    if e.zbc_cv(hw.Rng(s, n), curve["P"], curve["f"], n_steps_S1=500)["mom"] != want[s]:
                        errors.append(("zbc", s))
                    if not (e.bond_curve(hw.Rng(s, n))["P"] == wantc[s]).all():
                        errors.append(("curve", s))
            e.close()
        except Exception as exc:      # noqa: BLE001
            errors.append(repr(exc))

    ts = [threading.Thread(target=worker, args=(list(range(100 + 4 * k, 104 + 4 * k)),)) for k in range(2)]
    for t in ts:
        t.start()
    for t in ts:
        t.join()
    assert not errors, errors[:3]


def test_batches_longer_than_one_launch(engine, hw, curve):
    """more seeds than the 32-run seed axis of one launch: the batch entry points loop over launches"""
    n = 1 << 12
    seeds = [9000 + 7 * r for r in range(40)]
    res, _ = engine.zbc_cv_batch(seeds, n, curve["P"], curve["f"], n_steps_S1=500)
    vega, _ = engine.vega_pathwise_batch(seeds, n, curve["P"], curve["f"], n_steps_S1=500)
    assert len(res) == 40 and len(vega) == 40
    for r in (0, 31, 32, 39):
        one = engine.zbc_cv(hw.Rng(seeds[r], n), curve["P"], curve["f"], n_steps_S1=500)
        assert res[r]["mom"] == one["mom"] and res[r]["price_cv"] == one["price_cv"]
        pw = engine.vega_pathwise(hw.Rng(seeds[r], n), curve["P"], curve["f"], n_steps_S1=500)
        assert vega[r] == pw["vega_pathwise"]


def test_host_side_caches_follow_the_model(hw, curve):
    """the engine caches host-built tables (model arena, bumped-sigma FD arena) and the (int)(S1/dt) probe; every
    cache must be invalidated by a model change and keyed by its own arguments"""
    eng = hw.Engine(device=0)
    try:
        assert eng.steps_to(5.0) == 500 and eng.steps_to(5.0) == 500 and eng.steps_to(2.5) == 250
        fd1 = eng.vega_fd(hw.Rng(SEED, N), curve["P"], curve["f"], eps=0.001, n_steps_S1=500)
        fd2 = eng.vega_fd(hw.Rng(SEED, N), curve["P"], curve["f"], eps=0.002, n_steps_S1=500)
        fd1b = eng.vega_fd(hw.Rng(SEED, N), curve["P"], curve["f"], eps=0.001, n_steps_S1=500)
        assert fd1["price_minus"] == fd1b["price_minus"] and fd1["price_plus"] == fd1b["price_plus"]
        assert fd2["price_minus"] < fd1["price_minus"] < fd1["price_plus"] < fd2["price_plus"]
        # another model on the same engine: shorter grid, other sigma
        eng.set_model(hw.default_params(n_steps=200, n_mat=21, sigma=0.15))
        assert eng.steps_to(5.0) == 100
        c2 = eng.bond_curve(hw.Rng(SEED, N))
        fresh = hw.Engine(device=0, params=hw.default_params(n_steps=200, n_mat=21, sigma=0.15))
        c2f = fresh.bond_curve(hw.Rng(SEED, N))
        assert (c2["P"] == c2f["P"]).all()
        a = eng.vega_fd(hw.Rng(SEED, N), c2["P"], c2["f"], eps=0.001, n_steps_S1=100)
        b = fresh.vega_fd(hw.Rng(SEED, N), c2f["P"], c2f["f"], eps=0.001, n_steps_S1=100)
        assert a["price_minus"] == b["price_minus"] and a["price_plus"] == b["price_plus"]
        fresh.close()
        # and back: the default model's results are reproduced bit for bit
        eng.set_model(hw.default_params())
        assert eng.steps_to(5.0) == 500
        again = eng.vega_fd(hw.Rng(SEED, N), curve["P"], curve["f"], eps=0.001, n_steps_S1=500)
        assert again["price_minus"] == fd1["price_minus"] and again["price_plus"] == fd1["price_plus"]
    finally:
        eng.close()


def test_engine_lifecycle_and_argument_errors(hw, curve):
    """create/destroy repeatedly, bad arguments come back as status codes, never as a crash or exit()"""
    import ctypes as C
    lib = hw._ffi.load()
    free0 = torch.cuda.mem_get_info()[0]
    for k in range(6):
        e = hw.Engine(device=0)
        e.set_mode(k % 2)
        c = e.bond_curve(hw.Rng(k, 3000 + k))
        # P(0,0) = (2N) * MUFU.RCP((float)2N) like the reference's epilogue: exactly 1 only for powers of two
        assert abs(c["P"][0] - 1.0) < 2e-7 and np.isfinite(c["f"]).all()
        e.close()
    assert torch.cuda.mem_get_info()[0] > free0 - (64 << 20)          # nothing substantial leaked
    e = hw.Engine(device=0)
    try:
        assert lib.hw1f_bond_curve(e._h, None, None, None, None, None) == hw._ffi.ERR_INVALID
        assert lib.hw1f_engine_set_mode(e._h, 7) == hw._ffi.ERR_INVALID
        bad = hw.default_params(n_steps=1000, n_mat=77)                # 1000 % 76 != 0 (common.cuh:25-27)
        assert lib.hw1f_set_model(e._h, C.byref(bad)) == hw._ffi.ERR_INVALID
        assert b"divisible" in lib.hw1f_last_error(e._h)
        with pytest.raises(hw.HW1FError):
            e.sample_paths(hw.Rng(1, 8), 32)                           # more paths than the handle owns
        assert abs(e.bond_curve(hw.Rng(1, 777))["P"][0] - 1.0) < 2e-7  # still healthy
    finally:
        e.close()
    h = C.c_void_p()
    assert lib.hw1f_engine_create(99, C.byref(h)) == hw._ffi.ERR_NO_DEVICE


def test_bond_curve_submit_collect(engine, hw):
    """hw1f_bond_curve in two halves: several submissions in flight, collected out of order, bit-identical to the
    blocking call; slot misuse comes back as a status code"""
    seeds = [11, 12, 13, 14, 15, 16]
    want = [engine.bond_curve(hw.Rng(s, 5000 + 37 * s), timing=False) for s in seeds]
    slots = hw._ffi.ASYNC_SLOTS
    got = [None] * len(seeds)
    for k0 in range(0, len(seeds), slots):
        ks = list(range(k0, min(k0 + slots, len(seeds))))
        for k in ks:
            engine.set_model(engine.params)               # the per-call model upload of the reference's drivers
            engine.bond_curve_submit(hw.Rng(seeds[k], 5000 + 37 * seeds[k]), slot=k - k0)
        for k in reversed(ks):
            got[k] = engine.bond_curve_collect(slot=k - k0)
    for w, g in zip(want, got):
        for key in ("P", "f", "P_se"):
            assert (w[key] == g[key]).all(), key
    # a blocking call between submit and collect does not disturb the slot
    engine.bond_curve_submit(hw.Rng(seeds[0], 5000 + 37 * seeds[0]), slot=1)
    other = engine.bond_curve(hw.Rng(99, 4096), timing=False)
    again = engine.bond_curve_collect(slot=1)
    assert (again["P"] == want[0]["P"]).all() and not (other["P"][1:] == want[0]["P"][1:]).all()
    # a different model per call (one curve per sigma bump, src/3:449-482): every lane follows the caller's set_model
    base = engine.params
    sigmas = [0.08, 0.09, 0.1, 0.11, 0.12]
    try:
        blocking = []
        for sg in sigmas:
            engine.set_model(hw.default_params(sigma=sg))
            blocking.append(engine.bond_curve(hw.Rng(77, 6000), timing=False))
        lanes = [None] * len(sigmas)
        for k, sg in enumerate(sigmas):
            if k >= slots:
                lanes[k - slots] = engine.bond_curve_collect(slot=k % slots)
            engine.set_model(hw.default_params(sigma=sg))
            engine.bond_curve_submit(hw.Rng(77, 6000), slot=k % slots)
        for k in range(max(0, len(sigmas) - slots), len(sigmas)):
            lanes[k] = engine.bond_curve_collect(slot=k % slots)
        for b, l in zip(blocking, lanes):
            assert (b["P"] == l["P"]).all() and (b["f"] == l["f"]).all()
        assert not (blocking[0]["P"][1:] == blocking[-1]["P"][1:]).any()
    finally:
        engine.set_model(base)
    with pytest.raises(hw.HW1FError):
        engine.bond_curve_collect(slot=2)                 # nothing submitted
    engine.bond_curve_submit(hw.Rng(1, 2048), slot=0)
    with pytest.raises(hw.HW1FError):
        engine.bond_curve_submit(hw.Rng(2, 2048), slot=0)  # still in flight
    with pytest.raises(hw.HW1FError):
        engine.bond_curve_submit(hw.Rng(2, 2048), slot=slots)
    engine.bond_curve_collect(slot=0)
    # a fresh engine: the last slot first (its lane is created on demand), a model of another size is refused while a
    # submission is out, and destroying the engine with submissions in flight is clean
    e2 = hw.Engine(device=0)
    try:
        e2.set_mode(engine.mode)
        e2.bond_curve_submit(hw.Rng(5, 3000), slot=slots - 1)
        with pytest.raises(hw.HW1FError):
            e2.set_model(hw.default_params(n_steps=1000, n_mat=51))
        got3 = e2.bond_curve_collect(slot=slots - 1)
        assert (got3["P"] == engine.bond_curve(hw.Rng(5, 3000), timing=False)["P"]).all()
        e2.set_model(hw.default_params(n_steps=1000, n_mat=51))      # nothing in flight any more
        e2.bond_curve_submit(hw.Rng(6, 3000), slot=1)
        e2.bond_curve_submit(hw.Rng(7, 3000), slot=0)
        c51 = e2.bond_curve_collect(slot=1)
        assert c51["P"].shape == (51,) and abs(c51["P"][0] - 1.0) < 2e-7
    finally:
        e2.close()                                                   # slot 0 still in flight
