"""Engine vs the UNMODIFIED reference kernels run on a B200 with the same seeds.  This is the north-star
parity statement: integer RNG state bit-exact; P(0,T), theta, ZBC price, beta and vega within 1e-5
relative, or within the Monte Carlo CI where the reference's float-atomic summation dominates.

The reference outputs come from oracle/_ref/ref_harness when it is built (oracle/Makefile `ref`, which needs
the reference sources), else from tests/golden/ref_b200_seed20251018.json: the stored output of the same
`ref_harness parity 20251018` command on a B200."""
import json
import os
import subprocess

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HARNESS = os.path.join(ROOT, "oracle", "_ref", "ref_harness")
GOLDEN = os.path.join(ROOT, "tests", "golden", "ref_b200_seed20251018.json")
SEED = 20251018
N = 1 << 20


@pytest.fixture(scope="module")
def ref(tmp_path_factory):
    if not os.path.exists(HARNESS):
        with open(GOLDEN) as f:
            r = json.load(f)
        assert r["seed"] == SEED and r["n_paths"] == N
        return r
    out = tmp_path_factory.mktemp("ref") / "parity.json"
    subprocess.run([HARNESS, "parity", str(SEED), str(out)], check=True, stdout=subprocess.DEVNULL, timeout=600,
                   cwd=str(out.parent))
    with open(out) as f:
        r = json.load(f)
    keep = os.environ.get("HW1F_SAVE_REF")
    if keep:
        with open(keep, "w") as f:
            json.dump(r, f)
    return r


@pytest.fixture(scope="module")
def mine(engine, hw, ref):
    curve = engine.bond_curve(hw.Rng(SEED, N))
    return curve


def test_reference_rng_states_bit_exact(engine, hw, ref):
    rng = hw.Rng(SEED, N)
    for st in ref["states"]:
        state, _ = engine.debug_rng(rng, st["path"], 0)
        assert int(state[0]) == st["d"] and state[1:].tolist() == st["v"], st


def test_reference_curve(mine, ref, oracle):
    """The reference accumulates P_sum[m] with float32 atomics (market_data.cuh:63,73): 1024 block partials of ~2046
    are added to a running sum of ~2e6 whose ulp is 0.125.  At short maturities the partials are nearly identical, the
    rounding goes the same way at every add, and the error is a BIAS.  Measured on B200 (tests/parity_report.py ->
    profiles/r02_parity_report.json, same seeds on all sides): reference vs the double-precision oracle 1.01e-5 on P at
    T = 0.1 and 1.0e-4 on f(0,0), 1.05e-6 / 7e-6 for T >= 2, while two runs of the reference differ by 2.6e-7 / 2.3e-6
    (atomic reordering) and the engine sits on the oracle to 6.9e-8 / 1.1e-6.  Same seeds on both sides, so the Monte
    Carlo interval does not apply to the difference: the engine must sit on the exact (double) sum of the reference's
    own float paths, and the reference within 3x its own measured float-accumulation error of both."""
    P, f = np.array(ref["P"], np.float32), np.array(ref["f"], np.float32)
    P_orc, f_orc = oracle.bond_curve(SEED, N)            # full size: a few seconds on the box's cores
    assert np.abs(mine["P"] / P_orc - 1).max() < 3e-7     # measured 6.9e-8
    assert np.abs(mine["f"] - f_orc).max() < 4e-6         # measured 1.1e-6 / 1.5e-6 (both modes)
    assert np.abs(P / P_orc - 1).max() < 3e-5             # the reference's own float-atomic error: measured 1.01e-5
    assert np.abs(mine["P"] / P - 1).max() < 3e-5
    assert np.abs(mine["P"][20:] / P[20:] - 1).max() < 3e-6   # dispersed partials: measured 1.05e-6 (north star 1e-5)
    assert np.abs(mine["f"] - f).max() < 3e-4                 # f(0,0): measured 1.02e-4, all of it the reference's bias
    assert np.abs(mine["f"][20:] - f[20:]).max() < 2.2e-5     # measured 7.4e-6 (reference run to run: 2.3e-6)


def test_reference_theta(engine, mine, ref):
    got = engine.theta_calibrate(np.array(ref["f"], np.float32))
    assert np.abs(got["theta_rec"] - np.array(ref["theta_rec"], np.float32)).max() < 1e-6
    assert (got["theta_ref"] == np.array(ref["theta_orig"], np.float32)).all()


def test_reference_theta_end_to_end(engine, mine, ref, oracle):
    """the engine's OWN forward curve -> recover_theta against the reference's theta_rec (from its own curve).  theta
    differentiates f, so the reference's accumulation error enters 10x amplified: measured 7.3e-5 for T >= 2 and 1.2e-3
    at T = 0 (two runs of the reference differ by 1.4e-5); against the oracle chain (double sums of the same float paths
    -> f -> theta) the engine is within 3e-5."""
    th = engine.theta_calibrate(mine["f"])["theta_rec"]
    th_ref = np.array(ref["theta_rec"], np.float32)
    assert np.abs(th[20:] - th_ref[20:]).max() < 2.2e-4
    assert np.abs(th - th_ref).max() < 3.6e-3
    _, f_orc = oracle.bond_curve(SEED, N)
    th_orc = oracle.theta(f_orc)[0]
    assert np.abs(th - th_orc).max() < 6e-5                # f within 1.5e-6 of the oracle, differenced over 2 dT = 0.2 (0.1 at the ends)


def test_reference_zbc(engine, hw, ref):
    n_steps = engine.steps_to(5.0)
    P, f = np.array(ref["P"], np.float32), np.array(ref["f"], np.float32)
    z = engine.zbc_cv(hw.Rng(SEED + 54321, N), P, f, n_steps_S1=n_steps)
    # The reference output is one run, live or the stored one, and the reference is not deterministic (float atomics):
    # over 16 runs on one B200 (tools/ref_spread.py -> profiles/r02_ref_spread_16runs.json) its own beta* moves by 2.5e-5, rho by 1.2e-5, the
    # price by 1.3e-5 relative.  Worst engine-vs-run distance over those 16 runs, both modes: moments 1.0e-6, E[X] 8.1e-7,
    # price 1.5e-6, beta* 1.02e-5, rho 7.1e-6 (beta* and rho subtract nearly equal moments; medians 3.6e-6 / 2.1e-6).
    # Bounds = 4x the worst of 16 for the two quotients (a bound of 1e-5 failed one run in ~20), the north-star 1e-5 or
    # tighter for everything else.
    assert np.allclose(z["mom"], ref["zbc_moments"], rtol=1e-5)
    assert z["mean_X"] == pytest.approx(ref["zbc_mean_X"], rel=1e-5)
    assert z["price_cv"] == pytest.approx(ref["zbc_price_cv"], rel=6e-6)
    assert z["beta"] == pytest.approx(ref["zbc_beta"], rel=4e-5)
    assert z["corr"] == pytest.approx(ref["zbc_corr"], rel=3e-5)
    # ... and far inside the estimators' own standard errors (beta*: 1.2e-3 relative)
    assert abs(z["beta"] - ref["zbc_beta"]) < 0.05 * z["beta_se"]
    assert abs(z["corr"] - ref["zbc_corr"]) < 0.05 * z["corr_se"]
    assert abs(z["price_cv"] - ref["zbc_price_cv"]) < 0.05 * z["se_cv"]


def test_reference_vega(engine, hw, ref):
    n_steps = engine.steps_to(5.0)
    P, f = np.array(ref["P"], np.float32), np.array(ref["f"], np.float32)
    v = engine.vega(hw.Rng(SEED, N), P, f, n_steps_S1=n_steps)
    assert v["vega_pathwise"] == pytest.approx(ref["vega_pathwise"], rel=3e-6)    # measured 4.3e-7
    assert abs(v["vega_pathwise"] - ref["vega_pathwise"]) < 0.01 * v["vega_pathwise_se"]
    # FD quotients amplify float32 price rounding by 1/(2 eps) = 500.  Over 16 live runs of the reference
    # (profiles/r02_ref_spread_16runs.json): its own vega_fd moves by 6.1e-5, its vega_fd_recal by 2.9e-4 (the
    # recalibrated curves carry its float-atomic error of ~7e-6 on f(0,5), x 500); worst engine-vs-run distance 3.0e-5 /
    # 5.4e-4.  Bounds = 4x the worst of 16.
    assert v["vega_fd"] == pytest.approx(ref["vega_fd"], abs=1.2e-4)
    assert v["vega_fd_recal"] == pytest.approx(ref["vega_fd_recal"], abs=2.2e-3)


def test_reference_sample_paths(engine, hw, ref):
    got = engine.sample_paths(hw.Rng(SEED, N).seek(1000), 32)
    assert np.abs(got[0] - np.array(ref["r_path0"], np.float32)).max() < 2e-6
    assert np.abs(got[31] - np.array(ref["r_path31"], np.float32)).max() < 2e-6
