"""GPU parity tests proper: the CUDA engine (through the C ABI) against the CPU oracle on the same
seeded inputs.  Integer RNG work must be bit-exact; floating point follows BASELINE.json's
north_star tolerance (1e-5 relative for P, theta, ZBC price, beta, vega -- the engine/oracle gap
here is only the MUFU approximation error, so the tests use tighter bounds where they hold)."""
import json
import os

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

N = 1 << 13
SEED = 1234


@pytest.fixture(scope="module")
def curve(engine, hw):
    return engine.bond_curve(hw.Rng(SEED, N))


@pytest.fixture(scope="module")
def curve_ref(oracle):
    s, q = oracle.bond_curve_sums(SEED, N)
    P, f = oracle.curve_finalize(s, N)
    return s, q, P, f


# ---------------------------------------------------------------- integer layer: bit-exact
def test_rng_states_and_draws_bit_exact(engine, hw, oracle, golden_dir):
    with open(os.path.join(golden_dir, "xorwow_golden.json")) as f:
        golden = json.load(f)
    for c in golden["cases"]:
        if c["offset"] % 2 or c["subsequence"] >= (1 << 40):
            continue
        # handle window [subsequence - 3, subsequence + 5) so that hi/lo splitting is exercised
        first = max(c["subsequence"] - 3, 0)
        rng = hw.Rng(c["seed"], 8, first_path=first).seek(c["offset"])
        state, draws = engine.debug_rng(rng, c["subsequence"] - first, 2000)
        assert int(state[0]) == c["d"] and state[1:].tolist() == c["v"], c
        assert draws[:8].tolist() == c["draws_head"]
        assert int(draws[499]) == c["draw_499"] and int(draws[1999]) == c["draw_1999"]
        assert (draws == oracle.draws(c["seed"], c["subsequence"], c["offset"], 2000)).all()


@pytest.mark.parametrize("n_paths,first", [(1, 0), (31, 5), (513, 511), (4096, 0), (100000, 123457), (1 << 20, 0),
                                            (1 << 20, (1 << 30) - 512)])
def test_rng_any_geometry(engine, hw, oracle, n_paths, first):
    """ragged path ranges, unaligned first_path, chunk / hi-matrix boundaries"""
    rng = hw.Rng(987654321, n_paths, first_path=first)
    for q in sorted({0, n_paths // 2, n_paths - 1, min(511, n_paths - 1), min(512, n_paths - 1)}):
        state, draws = engine.debug_rng(rng, q, 12)
        assert (draws == oracle.draws(987654321, first + q, 0, 12)).all(), (n_paths, first, q)


def test_normals_match_device_formula(engine, hw, oracle):
    """Box-Muller floats: same uint32 inputs, MUFU vs libm in the transform"""
    for off in (0, 1, 500, 999):
        got = engine.debug_normals(hw.Rng(SEED, 64).seek(off), 17, 200)
        ref = oracle.normals(SEED, 17, off, 200)
        assert np.abs(got - ref).max() < 4e-6, off
    a = engine.debug_normals(hw.Rng(SEED, 64), 3, 100)
    b = engine.debug_normals(hw.Rng(SEED, 64).seek(37), 3, 63)
    assert (a[37:] == b).all()          # odd offsets land on the cached cos value, bit-exact


# ---------------------------------------------------------------- Q1
def test_bond_curve_vs_oracle(curve, curve_ref):
    s, q, P, f = curve_ref
    assert curve["P"][0] == 1.0
    assert np.abs(curve["P"] / P - 1).max() < 1e-6
    # f = -d ln P / dT: a 1e-7 relative wobble of P becomes ~5e-7 absolute in f (SURVEY 7.3-4)
    assert np.abs(curve["f"] - f).max() < 2e-6
    n = float(N)
    se = np.sqrt(np.maximum(q / 4 / n - (s / 2 / n) ** 2, 0) / n)
    assert np.allclose(curve["P_se"][1:], se[1:], rtol=2e-2, atol=1e-9)


def test_bond_curve_deterministic_and_offset(engine, hw, curve):
    again = engine.bond_curve(hw.Rng(SEED, N))
    assert (again["P"] == curve["P"]).all() and (again["f"] == curve["f"]).all()   # no atomics: bit-reproducible
    rng = hw.Rng(SEED, N)
    engine.bond_curve(rng)
    assert rng.tell() == 1000
    second = engine.bond_curve(rng)                      # normals [1000, 2000)
    assert rng.tell() == 2000 and not (second["P"] == curve["P"]).all()


def test_bond_curve_moments_shard_additivity(engine, hw):
    """sharding by path range is exact: moments([0,N)) == moments([0,a)) + moments([a,N)), ragged a"""
    import torch
    full = torch.zeros(202, dtype=torch.float64, device="cuda")
    a_ = torch.zeros(202, dtype=torch.float64, device="cuda")
    b_ = torch.zeros(202, dtype=torch.float64, device="cuda")
    cut = 5000 + 37
    torch.cuda.synchronize()
    engine.bond_curve_moments(hw.Rng(SEED, N), full.data_ptr())
    engine.bond_curve_moments(hw.Rng(SEED, cut), a_.data_ptr())
    engine.bond_curve_moments(hw.Rng(SEED, N - cut, first_path=cut), b_.data_ptr())
    engine.synchronize()
    # exact in exact arithmetic; the per-warp float shuffle trees see different groupings, so the
    # identity holds to float32 rounding of the (centred) warp sums
    assert torch.allclose(full[1:101], (a_ + b_)[1:101], rtol=2e-8, atol=0)
    assert torch.allclose(full[102:], (a_ + b_)[102:], rtol=2e-7, atol=0)
    out = engine.bond_curve_finish(full.data_ptr(), N)
    ref = engine.bond_curve(hw.Rng(SEED, N))
    assert (out["P"] == ref["P"]).all() and (out["f"] == ref["f"]).all()


def test_theta_vs_oracle(engine, oracle, curve):
    got = engine.theta_calibrate(curve["f"])
    rec, orig, Ts = oracle.theta(curve["f"])
    assert (got["T"] == Ts).all() and (got["theta_ref"] == orig).all()
    assert np.abs(got["theta_rec"] - rec).max() < 1e-6
    assert got["success"] == bool(np.abs(rec - orig)[::10].max() < 0.01)


# ---------------------------------------------------------------- Q2b / Q3
@pytest.mark.parametrize("n_steps,offset", [(500, 0), (499, 0), (500, 499), (499, 499), (500, 1000), (1, 0), (2, 3)])
def test_zbc_moments_vs_oracle(engine, hw, oracle, curve, n_steps, offset):
    rng = hw.Rng(SEED + 54321, N).seek(offset)
    got = engine.zbc_cv(rng, curve["P"], curve["f"], n_steps_S1=n_steps)
    assert rng.tell() == offset + n_steps
    mom = oracle.zbc_moments(SEED + 54321, N, curve["P"], curve["f"], n_steps_S1=n_steps, offset=offset)
    # after 1-2 steps every path sits at almost the same r, so P-K cancels ~150x and the MUFU.EX2
    # vs exp2f difference shows up coherently; with dispersed paths (>= 499 steps) it averages out
    rtol = 3e-6 if n_steps >= 499 else 2e-4
    assert np.allclose(got["mom"], mom, rtol=rtol), (got["mom"], mom)
    if n_steps >= 499:
        ref = oracle.zbc_algebra(got["mom"], 2 * N, float(curve["P"][100]))
        for k in ("mean_X", "mean_Y", "var_Y", "cov", "beta", "price_cv", "corr", "corr_single"):
            assert got[k] == pytest.approx(ref[k], rel=1e-6, abs=1e-12), k     # same float32 algebra
        assert got["ci95_lo"] < got["price_cv_f64"] < got["ci95_hi"]


def test_zbc_zero_steps_any_offset(engine, hw, oracle, curve):
    """n_steps_S1 == 0 (resolve_steps allows it): the payoff is evaluated at t = 0 whatever the parity of the
    normal offset -- an odd offset once consumed a Box-Muller pair and took one step (ADVICE r1)"""
    got = {}
    for offset in (0, 3):
        rng = hw.Rng(SEED + 54321, N).seek(offset)
        got[offset] = engine.zbc_cv(rng, curve["P"], curve["f"], n_steps_S1=0)
        assert rng.tell() == offset
        mom = oracle.zbc_moments(SEED + 54321, N, curve["P"], curve["f"], n_steps_S1=0, offset=offset)
        assert np.allclose(got[offset]["mom"], mom, rtol=2e-4), (got[offset]["mom"], mom)
    assert got[0]["mom"] == got[3]["mom"]
    v0 = engine.vega_pathwise(hw.Rng(SEED, N), curve["P"], curve["f"], n_steps_S1=0)
    v1 = engine.vega_pathwise(hw.Rng(SEED, N).seek(1), curve["P"], curve["f"], n_steps_S1=0)
    assert v0["vega_pathwise_f64"] == v1["vega_pathwise_f64"]


def test_zbc_steps_probe(engine):
    n = engine.steps_to(5.0)
    assert n in (499, 500)
    assert engine.steps_to(10.0) in (999, 1000)


def test_vega_pathwise_vs_oracle(engine, hw, oracle, curve):
    for n_steps, offset in ((500, 0), (499, 1)):
        got = engine.vega_pathwise(hw.Rng(SEED, N).seek(offset), curve["P"], curve["f"], n_steps_S1=n_steps)
        s, q = oracle.vega_pathwise_sums(SEED, N, curve["P"], curve["f"], n_steps_S1=n_steps, offset=offset)
        assert got["vega_pathwise_f64"] == pytest.approx(s / N, rel=5e-6)
        se = np.sqrt((q / N - (s / N) ** 2) / N)
        assert got["vega_pathwise_se"] == pytest.approx(se, rel=1e-3)


def test_vega_fd_vs_oracle(engine, hw, oracle, curve):
    """both bumps in one launch == two oracle runs on the same normals with shifted drift tables"""
    eps, sig = np.float32(0.001), np.float32(0.1)
    rng = hw.Rng(SEED, N).seek(500)
    got = engine.vega_fd(rng, curve["P"], curve["f"], eps=float(eps), n_steps_S1=500)
    assert rng.tell() == 1000
    prices = []
    for s_new in (sig - eps, sig + eps):
        drift = oracle.shifted_drift_table(float(s_new))
        assert (drift == engine.drift_table(2, float(s_new))).all()
        mom = oracle.zbc_moments(SEED, N, curve["P"], curve["f"], n_steps_S1=500, offset=500, sigma=float(s_new),
                                 drift=drift)
        prices.append(oracle.zbc_algebra(mom, 2 * N, float(curve["P"][100]))["price_cv"])
    assert got["price_minus"] == pytest.approx(prices[0], rel=2e-5)
    assert got["price_plus"] == pytest.approx(prices[1], rel=2e-5)
    # the difference quotient amplifies price noise by 1/(2 eps) = 500
    assert got["vega_fd"] == pytest.approx((prices[1] - prices[0]) / (2 * float(eps)), abs=2e-3)


@pytest.mark.parametrize("n_steps", [500, 490, 495])
def test_vega_fd_recalibrated_vs_oracle(engine, hw, oracle, n_steps):
    """n_steps on the maturity grid (500, 490): decomposed mode prices from the noise state the curve pass parked
    (one simulation); 495: off the grid, second pass over the same normals; reference-order mode: always two passes"""
    eps, sig = np.float32(0.001), np.float32(0.1)
    rng = hw.Rng(SEED, N).seek(1000)
    got = engine.vega_fd_recalibrated(rng, eps=float(eps), n_steps_S1=n_steps)
    assert rng.tell() == 1000 + n_steps
    prices = []
    for s_new in (sig - eps, sig + eps):
        sums, _ = oracle.bond_curve_sums(SEED, N, offset=1000, sigma=float(s_new))     # unshifted base drift
        P, f = oracle.curve_finalize(sums, N)
        mom = oracle.zbc_moments(SEED, N, P, f, n_steps_S1=n_steps, offset=1000, sigma=float(s_new))
        prices.append(oracle.zbc_algebra(mom, 2 * N, float(P[100]))["price_cv"])
    assert got["price_minus_recal"] == pytest.approx(prices[0], rel=5e-5)
    assert got["price_plus_recal"] == pytest.approx(prices[1], rel=5e-5)


@pytest.mark.parametrize("over,S1,S2", [
    (dict(), 2.0, 7.0),                                   # windows in the middle of the grid
    (dict(), 0.1, 0.3),                                   # left edge: the S1 window starts at grid point 0
    (dict(), 9.0, 10.0),                                  # both windows at the right edge
    (dict(n_steps=240, n_mat=13, T_final=2.4), 1.0, 2.0),  # a 13-point grid: the windows cover most of it
])
def test_vega_fd_recalibrated_sparse_save_points(engine, hw, over, S1, S2):
    """the one-pass recalibration evaluates only the save points its pricing reads (two windows around S1 and S2 and
    the last maturity, fast_kernel DUMP): same prices as full curves from engines whose model carries the bumped sigma"""
    eps, n = 0.001, 1 << 13
    e1 = hw.Engine(device=0, params=hw.default_params(**over))
    e1.set_mode(engine.mode)
    try:
        ns = e1.steps_to(S1)
        if ns % e1.constants.save_stride:
            ns -= ns % e1.constants.save_stride            # on the maturity grid: the one-pass route
        c0 = e1.bond_curve(hw.Rng(9, n))
        nm = e1.n_mat
        K = float(np.float32(0.9) * c0["P"][int(round(S2 / e1.constants.mat_spacing))] /
                  c0["P"][int(round(S1 / e1.constants.mat_spacing))])
        got = e1.vega_fd_recalibrated(hw.Rng(SEED, n).seek(1000), eps=eps, S1=S1, S2=S2, K=K, n_steps_S1=ns)
        prices = []
        for sgn in (-1.0, 1.0):
            sg = float(np.float32(e1.params.sigma) + np.float32(sgn * eps))
            e2 = hw.Engine(device=0, params=hw.default_params(sigma=sg, **over))
            e2.set_mode(engine.mode)
            c = e2.bond_curve(hw.Rng(SEED, n).seek(1000))
            z = e2.zbc_cv(hw.Rng(SEED, n).seek(1000), c["P"], c["f"], S1=S1, S2=S2, K=K, n_steps_S1=ns)
            prices.append(z["price_cv"])
            e2.close()
        assert nm == len(c["P"])
        assert got["price_minus_recal"] == pytest.approx(prices[0], rel=3e-6)
        assert got["price_plus_recal"] == pytest.approx(prices[1], rel=3e-6)
    finally:
        e1.close()


def test_vega_fd_recalibrated_equals_bumped_engines(engine, hw):
    """recompute_market_data + run_zbc_price at sigma -/+ eps (src/3:449-525) composed from the public single-scenario
    calls on engines whose MODEL carries the bumped sigma (the base drift does not depend on sigma): the fused
    two-scenario launches of hw1f_vega_fd_recalibrated must give the same prices"""
    eps = 0.001
    got = engine.vega_fd_recalibrated(hw.Rng(SEED, N).seek(1000), eps=eps, n_steps_S1=500)
    prices = []
    for sgn in (-1.0, 1.0):
        e2 = hw.Engine(device=0, params=hw.default_params(sigma=float(np.float32(0.1) + np.float32(sgn * eps))))
        e2.set_mode(engine.mode)
        c = e2.bond_curve(hw.Rng(SEED, N).seek(1000))
        z = e2.zbc_cv(hw.Rng(SEED, N).seek(1000), c["P"], c["f"], n_steps_S1=500)
        prices.append(z["price_cv"])
        e2.close()
    assert got["price_minus_recal"] == pytest.approx(prices[0], rel=2e-6)
    assert got["price_plus_recal"] == pytest.approx(prices[1], rel=2e-6)


@pytest.mark.parametrize("n", [500, 499, 250])
def test_vega_sequence_windows(engine, hw, curve, n):
    """hw1f_vega walks the reference's draw windows: [0,n) pathwise, [n,2n) FD, [2n,..) recalibrated (odd n: the FD
    window starts on the cos half of a Box-Muller pair, the recalibrated prices take the second pass)"""
    rng = hw.Rng(SEED, N)
    allres = engine.vega(rng, curve["P"], curve["f"], n_steps_S1=n)
    assert rng.tell() == 3 * n
    pw = engine.vega_pathwise(hw.Rng(SEED, N), curve["P"], curve["f"], n_steps_S1=n)
    fd = engine.vega_fd(hw.Rng(SEED, N).seek(n), curve["P"], curve["f"], n_steps_S1=n)
    rc = engine.vega_fd_recalibrated(hw.Rng(SEED, N).seek(2 * n), n_steps_S1=n)
    assert allres["vega_pathwise"] == pw["vega_pathwise"]
    assert allres["vega_fd"] == fd["vega_fd"] and allres["vega_fd_recal"] == rc["vega_fd_recal"]
    if n == 500:
        assert 0.05 < allres["vega_pathwise"] < 0.5 and 0.05 < allres["vega_fd"] < 0.5    # src/3:789-790


def test_vega_sequence_first_call_on_a_fresh_engine(engine, hw, curve):
    """hw1f_vega as the FIRST pricing call of an engine (no bumped-sigma arena yet, ragged path count) equals the
    three separate calls on another fresh engine"""
    n = (1 << 12) + 77
    a = hw.Engine(device=0)
    a.set_mode(engine.mode)
    got = a.vega(hw.Rng(SEED, n), curve["P"], curve["f"], n_steps_S1=500)
    a.close()
    b = hw.Engine(device=0)
    b.set_mode(engine.mode)
    pw = b.vega_pathwise(hw.Rng(SEED, n), curve["P"], curve["f"], n_steps_S1=500)
    fd = b.vega_fd(hw.Rng(SEED, n).seek(500), curve["P"], curve["f"], n_steps_S1=500)
    rc = b.vega_fd_recalibrated(hw.Rng(SEED, n).seek(1000), n_steps_S1=500)
    b.close()
    assert got["vega_pathwise"] == pw["vega_pathwise"]
    assert got["price_minus"] == fd["price_minus"] and got["price_plus"] == fd["price_plus"]
    assert got["price_minus_recal"] == rc["price_minus_recal"] and got["price_plus_recal"] == rc["price_plus_recal"]


@pytest.mark.parametrize("n", [1, 2, 33, 1023, 1025])
def test_tiny_and_ragged_path_counts(engine, hw, oracle, curve, n):
    """a single subsequence, less than a warp, one short of / one past a chunk: masks and reductions at the edges"""
    c = engine.bond_curve(hw.Rng(SEED, n, first_path=7))
    s, _ = oracle.bond_curve_sums(SEED, n, first_path=7)
    P, f = oracle.curve_finalize(s, n)
    assert np.abs(c["P"] / P - 1).max() < 1e-6 and np.abs(c["f"] - f).max() < 5e-6
    z = engine.zbc_cv(hw.Rng(SEED, n, first_path=7), curve["P"], curve["f"], n_steps_S1=500)
    mom = oracle.zbc_moments(SEED, n, curve["P"], curve["f"], n_steps_S1=500, first_path=7)
    # a handful of paths: no averaging of the per-path MUFU-vs-libm differences (the payoff P - K ~ 0.02 amplifies
    # the 1e-7 of P forty-fold)
    assert np.allclose(z["mom"], mom, rtol=(2e-5 if n < 64 else 5e-6), atol=1e-12)
    fu = engine.fused(hw.Rng(SEED, n, first_path=7), curve["P"], curve["f"], n_steps_S1=500)
    assert (fu["P"] == c["P"]).all() and fu["zbc"]["mom"] == z["mom"]


@pytest.mark.parametrize("n_steps", [1000, 998, 2])
def test_zbc_at_the_ends_of_the_grid(engine, hw, oracle, curve, n_steps):
    """S1 at the last step of the model, and a two-step option.  The two-step call is far out of the money
    (P(0.02,10) ~ 0.86 < K = 0.905): only a few paths pay, each by P - K ~ 1e-5, so the X sums are conditioned like
    1e-7 / 1e-5 -- they are compared at 1e-4, the control-variate sums (no kink) at the usual 5e-6"""
    S1 = n_steps * 0.01
    z = engine.zbc_cv(hw.Rng(SEED, N), curve["P"], curve["f"], S1=S1, S2=10.0, n_steps_S1=n_steps)
    mom = oracle.zbc_moments(SEED, N, curve["P"], curve["f"], S1=S1, S2=10.0, n_steps_S1=n_steps)
    got = np.asarray(z["mom"])
    assert np.allclose(got[[1, 3]], mom[[1, 3]], rtol=5e-6)
    assert np.allclose(got[[0, 2, 4]], mom[[0, 2, 4]], rtol=(1e-4 if n_steps == 2 else 5e-6), atol=1e-12)


def test_huge_offsets_and_path_indices(engine, hw, oracle, curve):
    """normal offsets beyond 32 bits (the Weyl word wraps, T^offset comes from the host jump tables) and path
    indices just below the 2^41 limit of the window tables"""
    for first, off in ((0, (1 << 36) + 2), ((1 << 41) - 5000, 0), ((1 << 40) + 3, (1 << 33) + 4)):
        n = 700
        st, draws = engine.debug_rng(hw.Rng(SEED, n, first_path=first).seek(off), 699, 6)
        assert (draws == oracle.draws(SEED, first + 699, 2 * (off // 2), 6)).all(), (first, off)
        c = engine.bond_curve(hw.Rng(SEED, n, first_path=first).seek(off))
        s, _ = oracle.bond_curve_sums(SEED, n, first_path=first, offset=off)
        P, f = oracle.curve_finalize(s, n)
        assert np.abs(c["P"] / P - 1).max() < 1e-6, (first, off)
    with pytest.raises(hw.HW1FError):
        engine.bond_curve(hw.Rng(SEED, 10, first_path=(1 << 42)))


def test_batches_equal_single_runs(engine, hw, curve):
    seeds = [1700000000000000 + r * 12345 for r in range(5)]            # src/2:223-229
    res, _ = engine.zbc_cv_batch(seeds, N, curve["P"], curve["f"], n_steps_S1=500)
    for s, r in zip(seeds, res):
        one = engine.zbc_cv(hw.Rng(s, N), curve["P"], curve["f"], n_steps_S1=500)
        assert r["mom"] == one["mom"] and r["price_cv"] == one["price_cv"]
    vseeds = [3400000000 + r * 982451653 for r in range(4)]               # src/3:539-545
    vega, _ = engine.vega_pathwise_batch(vseeds, N, curve["P"], curve["f"], n_steps_S1=500)
    for s, v in zip(vseeds, vega):
        assert v == engine.vega_pathwise(hw.Rng(s, N), curve["P"], curve["f"], n_steps_S1=500)["vega_pathwise"]


def test_sample_paths_vs_oracle(engine, hw, oracle):
    rng = hw.Rng(SEED, N).seek(1000)                    # the reference dumps draws 1000..1999 (src/1:163)
    got = engine.sample_paths(rng, 32)
    ref = oracle.sample_paths(SEED, 32, offset=1000)
    assert rng.tell() == 1000                           # no write-back (market_data.cuh:159)
    assert got.shape == (32, 1001) and np.abs(got - ref).max() < 2e-6


def test_errors_are_reported_not_fatal(engine, hw, curve):
    with pytest.raises(hw.HW1FError):
        engine.zbc_cv(hw.Rng(1, N), curve["P"], curve["f"], n_steps_S1=5000)
    with pytest.raises(hw.HW1FError):
        engine.bond_curve(hw.Rng(1, N).seek(1))         # odd offset: documented as unsupported for Q1
    assert engine.bond_curve(hw.Rng(SEED, N))["P"][0] == 1.0     # engine still usable


# ---------------------------------------------------------------- full size: size-independent properties
def test_full_size_closed_form(engine, hw):
    n = 1 << 20
    c = engine.bond_curve(hw.Rng(20240101, n))
    assert abs(c["P"][50] - 0.947126) < 5 * c["P_se"][50] + 1e-5
    assert abs(c["P"][100] - 0.859387) < 5 * c["P_se"][100] + 1e-5
    z = engine.zbc_cv(hw.Rng(20240101 + 54321, n), c["P"], c["f"])
    assert abs(z["price_cv_f64"] - 0.025255) < 6 * z["se_cv"] + 2e-5
    assert abs(z["mean_Y"] - c["P"][100]) < 1e-3
    v = engine.vega_pathwise(hw.Rng(7, n), c["P"], c["f"])
    assert abs(v["vega_pathwise_f64"] - 0.240) < 5 * v["vega_pathwise_se"] + 2e-3


def test_grid_stride_chunks_large_run(engine, hw, curve):
    """more chunks than resident blocks: blocks stride over chunks and fold them into their double
    accumulators; the result must equal the sum of shards that each fit in one pass"""
    import torch
    grid = 32 * torch.cuda.get_device_properties(0).multi_processor_count      # prepare_launch's grid cap
    n = (2 * grid + 37) * 1024 + 3            # chunks of kChunk = 1024 subsequences
    n_chunks = (n + 1023) // 1024
    assert n_chunks > 2 * grid                # every block folds 2 or 3 chunks
    counts = [grid * 1024, grid * 1024, n - 2 * grid * 1024]     # shards of <= grid chunks: one pass each
    assert all((c + 1023) // 1024 <= grid for c in counts)
    full = torch.zeros(202, dtype=torch.float64, device="cuda")
    torch.cuda.synchronize()
    engine.bond_curve_moments(hw.Rng(99, n), full.data_ptr())
    acc = torch.zeros(202, dtype=torch.float64, device="cuda")
    part = torch.zeros(202, dtype=torch.float64, device="cuda")
    torch.cuda.synchronize()
    first = 0
    for cnt in counts:
        engine.bond_curve_moments(hw.Rng(99, cnt, first_path=first), part.data_ptr())
        engine.synchronize()
        acc += part
        torch.cuda.synchronize()
        first += cnt
    assert torch.allclose(full[1:101], acc[1:101], rtol=2e-8, atol=0)
    assert torch.allclose(full[102:], acc[102:], rtol=2e-7, atol=0)
    # same for the ZBC moments (double all the way: tight)
    zf = torch.zeros(5, dtype=torch.float64, device="cuda")
    za = torch.zeros(5, dtype=torch.float64, device="cuda")
    zp = torch.zeros(5, dtype=torch.float64, device="cuda")
    torch.cuda.synchronize()
    engine.zbc_cv_moments(hw.Rng(99, n), curve["P"], curve["f"], zf.data_ptr(), n_steps_S1=500)
    first = 0
    for cnt in counts:
        engine.zbc_cv_moments(hw.Rng(99, cnt, first_path=first), curve["P"], curve["f"], zp.data_ptr(), n_steps_S1=500)
        engine.synchronize()
        za += zp
        torch.cuda.synchronize()
        first += cnt
    assert torch.allclose(zf, za, rtol=1e-12, atol=0)


@pytest.mark.parametrize("over", [
    dict(n_steps=200, n_mat=21),                                   # stride 10, short grid
    dict(n_steps=400, n_mat=101),                                  # stride 4: remainder pairs in the 5-pair unroll
    dict(n_steps=600, n_mat=51, T_final=6.0),                      # stride 12, dt = 0.01, spacing 0.12
    dict(a=0.5, sigma=0.2, r0=0.03, theta_a0=0.02, theta_b0=0.001, theta_a1=0.03, theta_b1=-0.0005, theta_break=4.0),
    # weak mean reversion: 1 - e^{-a dt} = 5e-4, the decomposed kernels' q = qA W - qB h has qA = 4000
    dict(a=0.05, sigma=0.02, r0=0.02),
    # ODD save strides (the reference's configuration space, common.cuh:25-29): save points fall between the two
    # normals of a Box-Muller pair
    dict(n_steps=500, n_mat=101),                                  # stride 5
    dict(n_steps=700, n_mat=101, T_final=7.0),                     # stride 7
    dict(n_steps=55, n_mat=12, T_final=5.5),                       # stride 5, ODD step count: the curve ends mid-pair
    # the ends of the configuration space hw1f_set_model accepts (n_mat in [3, 1024], n_steps in [2, 8192])
    dict(n_steps=2, n_mat=3, T_final=0.5),                         # two steps, stride 1: every step is a save point
    dict(n_steps=8184, n_mat=1024),                                # 1024 maturities (2048 curve slots per block), stride 8
    dict(n_steps=1023, n_mat=1024, T_final=10.23),                 # stride 1 on the longest grid
])
@pytest.mark.parametrize("mode", [0, 1])
def test_other_model_parameters(hw, over, mode):
    """the engine is not specialised to the reference's macros (common.cuh:16-39)"""
    from oracle_lib import Oracle
    o = Oracle(**over)
    eng = hw.Engine(device=0, params=hw.default_params(**over))
    eng.set_mode(mode)
    try:
        n = 1 << 12
        c = eng.bond_curve(hw.Rng(31337, n))
        P, f = o.bond_curve(31337, n)
        # f differences ln P over one grid spacing: one float32 ulp of P (6e-8) is worth 6e-8 / spacing in f
        f_tol = max(5e-6, 2 * 6e-8 * (o.p.n_mat - 1) / o.p.T_final)
        assert np.abs(c["P"] / P - 1).max() < 1e-6 and np.abs(c["f"] - f).max() < f_tol
        assert (eng.drift_table(0) == o.drift_tables()[0]).all() and (eng.drift_table(1) == o.drift_tables()[1]).all()
        th = eng.theta_calibrate(c["f"])
        assert np.abs(th["theta_rec"] - o.theta(c["f"])[0]).max() < 2e-6
        S1, S2 = 0.4 * o.p.T_final, 0.8 * o.p.T_final
        ns = eng.steps_to(S1)
        assert abs(ns - S1 / o.dt) <= 1
        K = float(np.float32(0.9) * P[int(round(0.8 * (o.p.n_mat - 1)))] / P[int(round(0.4 * (o.p.n_mat - 1)))])
        z = eng.zbc_cv(hw.Rng(5, n), c["P"], c["f"], S1=S1, S2=S2, K=K, n_steps_S1=ns)
        mom = o.zbc_moments(5, n, c["P"], c["f"], S1=S1, S2=S2, K=K, n_steps_S1=ns)
        assert np.allclose(z["mom"], mom, rtol=5e-6)
        v = eng.vega_pathwise(hw.Rng(6, n), c["P"], c["f"], S1=S1, S2=S2, K=K, n_steps_S1=ns)
        s, _ = o.vega_pathwise_sums(6, n, c["P"], c["f"], S1=S1, S2=S2, K=K, n_steps_S1=ns)
        assert v["vega_pathwise_f64"] == pytest.approx(s / n, rel=2e-5, abs=1e-7)
    finally:
        eng.close()


@pytest.mark.parametrize("mode", [0, 1])
def test_odd_save_stride_q3_and_offsets(hw, mode):
    """stride 5 (500 steps on 101 maturities): hw1f_vega takes the three-call route, the recalibrated FD its second
    pass, and every estimator equals an engine whose curve inputs come from the oracle-checked path; a curve over an ODD
    number of steps leaves the handle mid-pair and the next launch picks up the cached cos normal"""
    from oracle_lib import Oracle
    over = dict(n_steps=500, n_mat=101)
    o = Oracle(**over)
    eng = hw.Engine(device=0, params=hw.default_params(**over))
    eng.set_mode(mode)
    try:
        n = 1 << 12
        c = eng.bond_curve(hw.Rng(777, n))
        P, f = o.bond_curve(777, n)
        assert np.abs(c["P"] / P - 1).max() < 1e-6 and np.abs(c["f"] - f).max() < 5e-6
        ns = eng.steps_to(5.0)
        assert ns == 250
        rng = hw.Rng(778, n)
        v = eng.vega(rng, c["P"], c["f"], n_steps_S1=ns)
        assert rng.tell() == 3 * ns
        pw = eng.vega_pathwise(hw.Rng(778, n), c["P"], c["f"], n_steps_S1=ns)
        fd = eng.vega_fd(hw.Rng(778, n).seek(ns), c["P"], c["f"], n_steps_S1=ns)
        rc = eng.vega_fd_recalibrated(hw.Rng(778, n).seek(2 * ns), n_steps_S1=ns)
        assert v["vega_pathwise"] == pw["vega_pathwise"] and v["vega_fd"] == fd["vega_fd"]
        assert v["vega_fd_recal"] == rc["vega_fd_recal"]
        s, _ = o.vega_pathwise_sums(778, n, c["P"], c["f"], n_steps_S1=ns)
        assert v["vega_pathwise_f64"] == pytest.approx(s / n, rel=2e-5, abs=1e-7)
        # recalibrated prices against the oracle: curves at sigma -/+ eps on normals [2 ns, 2 ns + 500), prices on [2 ns, 3 ns)
        eps, sig = np.float32(0.001), np.float32(0.1)
        prices = []
        for sg in (sig - eps, sig + eps):
            sums, _ = o.bond_curve_sums(778, n, offset=2 * ns, sigma=float(sg))     # unshifted base drift
            Pb, fb = o.curve_finalize(sums, n)
            mom = o.zbc_moments(778, n, Pb, fb, n_steps_S1=ns, offset=2 * ns, sigma=float(sg))
            prices.append(o.zbc_algebra(mom, 2 * n, float(Pb[-1]))["price_cv"])
        assert v["price_minus_recal"] == pytest.approx(prices[0], rel=5e-5)
        assert v["price_plus_recal"] == pytest.approx(prices[1], rel=5e-5)
    finally:
        eng.close()
    # odd step count: 55 steps -> the handle sits on an odd offset; sample paths continue from the cached cos normal
    over = dict(n_steps=55, n_mat=12, T_final=5.5)
    o = Oracle(**over)
    eng = hw.Engine(device=0, params=hw.default_params(**over))
    eng.set_mode(mode)
    try:
        rng = hw.Rng(779, 64)
        eng.bond_curve(rng)
        assert rng.tell() == 55
        got = eng.sample_paths(rng, 8)
        want = o.sample_paths(779, 8, offset=55)
        assert np.abs(got - want).max() < 2e-6
        with pytest.raises(hw.package.engine.HW1FError):      # a second curve would have to start mid-pair
            eng.bond_curve(rng)
    finally:
        eng.close()


def test_far_subsequences_and_offsets(engine, hw, oracle, curve):
    """path ranges far from 0 (hi part of the jump tables) and large normal offsets (T^offset folded on the host)"""
    first, n = (1 << 33) + 12345, 3000
    c = engine.bond_curve(hw.Rng(SEED, n, first_path=first).seek(100000))
    s, _ = oracle.bond_curve_sums(SEED, n, first_path=first, offset=100000)
    P, f = oracle.curve_finalize(s, n)
    assert np.abs(c["P"] / P - 1).max() < 1e-6 and np.abs(c["f"] - f).max() < 5e-6
    z = engine.zbc_cv(hw.Rng(SEED, n, first_path=first).seek(1000001), curve["P"], curve["f"], n_steps_S1=499)
    mom = oracle.zbc_moments(SEED, n, curve["P"], curve["f"], n_steps_S1=499, first_path=first, offset=1000001)
    assert np.allclose(z["mom"], mom, rtol=5e-6)
