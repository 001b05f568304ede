"""The cap / floor strip kernel (cap_kernel) at the edges of its schedule, geometry and model space, in both arithmetic
modes: every segment length of the walk between reset steps (and so every split of the decomposed mode into 5-pair
groups and single pairs), shared reset steps, every normal-offset parity, ragged path ranges, odd strides and step
counts, weak mean reversion, the 100-caplet maximum on the longest grid, degenerate caplets, the host algebra and the
state an engine carries across calls."""
import numpy as np
import pytest

import cap_oracle
from cap_closed_form import atm_rate, interp_mkt

pytestmark = pytest.mark.gpu

N = 1 << 13
SEED = 2718


@pytest.fixture(scope="module")
def curve(engine, hw):
    return engine.bond_curve(hw.Rng(SEED, N))


def schedule(hw, steps, dt, T_final, P, tau=0.25):
    steps = np.asarray(steps)
    resets = steps * dt
    pays = np.minimum(resets + tau, T_final)
    caps = hw.caplet_schedule(resets, pays, atm_rate(P, resets, pays, T_final))
    caps["n_steps_reset"] = steps
    return caps


def all_moments(res):
    return np.vstack([res["mom"], np.asarray(res["strip"]["mom"])[None, :]])


def check(got, ref, rel=3e-6, what=""):
    mom = all_moments(got)
    gap, bound = np.abs(mom - ref), cap_oracle.moment_bound(ref, rel=rel)
    print(f"{what}: worst moment gap / bound {(gap / bound).max():.3g}")
    assert np.isfinite(mom).all()
    assert (gap <= bound).all(), (what, np.unravel_index((gap / bound).argmax(), gap.shape), (gap / bound).max())


# ---------------------------------------------------------------- 1. segment shapes
# from step 1, gaps 1, 2, 3, 4, 5, 6, 7, 9, 10, 11, 0 (two caplets on one step), 13, then one long segment to a late
# step: segments that start and end on either parity, so every split into 5-pair groups plus single pairs (decomposed
# mode) and a cached cos half at either end of a segment
SEG_STEPS = np.cumsum([1, 1, 2, 3, 4, 5, 6, 7, 9, 10, 11, 0, 13]).tolist() + [901]


@pytest.mark.parametrize("kind", ["cap", "floor"])
@pytest.mark.parametrize("offset", [0, 1, 2, 3])
def test_segment_shapes_vs_oracle(engine, hw, oracle, curve, kind, offset):
    caps = schedule(hw, SEG_STEPS, 0.01, 10.0, curve["P"])
    rng = hw.Rng(SEED + 1, N).seek(offset)
    got = engine.cap_floor(rng, caps, curve["P"], curve["f"], kind=kind)
    assert rng.tell() == offset + SEG_STEPS[-1]
    ref = cap_oracle.cap_moments(oracle, SEED + 1, N, caps, curve["P"], curve["f"], kind=kind, offset=offset)
    check(got, ref, what=f"{kind} offset {offset}")


# ---------------------------------------------------------------- 2. ragged geometry
@pytest.mark.parametrize("n", [1, 2, 33, 1023, 1025])
def test_ragged_path_counts_vs_oracle(engine, hw, oracle, curve, n):
    caps = schedule(hw, SEG_STEPS, 0.01, 10.0, curve["P"])
    got = engine.cap_floor(hw.Rng(SEED + 2, n, first_path=7).seek(1), caps, curve["P"], curve["f"], kind="cap")
    ref = cap_oracle.cap_moments(oracle, SEED + 2, n, caps, curve["P"], curve["f"], kind="cap", first_path=7, offset=1)
    # below 64 paths the per-path MUFU-vs-libm differences of the controls do not average out: the allowance of
    # test_tiny_and_ragged_path_counts (2e-5 instead of the usual bound)
    check(got, ref, rel=(2e-5 if n < 64 else 3e-6), what=f"n = {n}")


# ---------------------------------------------------------------- 3. models
MODELS = [
    dict(n_steps=400, n_mat=101),                       # stride 4
    dict(n_steps=500, n_mat=101),                       # stride 5: save points fall inside a Box-Muller pair
    dict(n_steps=700, n_mat=101, T_final=7.0),          # stride 7
    dict(n_steps=200, n_mat=21),                        # stride 10
    dict(n_steps=55, n_mat=12, T_final=5.5),            # odd step count
    dict(n_steps=2, n_mat=3, T_final=0.5),              # two steps: one caplet at step 1, paid at T_final
    dict(a=0.05, sigma=0.02, r0=0.02),                  # weak mean reversion: the decomposed I rebuild has qA = 4000
    dict(n_steps=1023, n_mat=1024, T_final=10.23),      # stride 1 on the longest grid
]


@pytest.mark.parametrize("over", MODELS, ids=lambda o: "-".join(f"{k}{v}" for k, v in o.items()))
def test_models_vs_oracle(engine, hw, over):
    from oracle_lib import Oracle
    o = Oracle(**over)
    eng = hw.Engine(device=0, params=hw.default_params(**over))
    eng.set_mode(engine.mode)
    try:
        n, ns, Tf = 1 << 12, eng.n_steps, float(eng.params.T_final)
        c = eng.bond_curve(hw.Rng(31337, n))
        steps = [1] if ns == 2 else np.unique(np.linspace(1, 0.8 * ns, 9).round().astype(int))
        caps = schedule(hw, steps, Tf / ns, Tf, c["P"], tau=(0.25 if ns == 2 else 0.2 * Tf))
        for kind, off in (("cap", 0), ("floor", 1)):
            got = eng.cap_floor(hw.Rng(5, n).seek(off), caps, c["P"], c["f"], kind=kind)
            ref = cap_oracle.cap_moments(o, 5, n, caps, c["P"], c["f"], kind=kind, offset=off)
            # 5e-6: test_other_model_parameters' bound for these models at 4096 paths
            check(got, ref, rel=5e-6, what=f"{over} {kind}")
    finally:
        eng.close()


def test_hundred_caplets_on_the_longest_grid(engine, hw):
    """HW1F_MAX_CAPLETS on 8184 steps: the largest shared-memory footprint (reference order stages the drift of every
    step up to the last reset, ~85 KB).  It must price; a refusal would be HW1F_ERR_UNSUPPORTED, never a wrong number."""
    from oracle_lib import Oracle
    over = dict(n_steps=8184, n_mat=1024)
    o = Oracle(**over)
    eng = hw.Engine(device=0, params=hw.default_params(**over))
    eng.set_mode(engine.mode)
    try:
        n, ns, Tf = 1 << 12, eng.n_steps, float(eng.params.T_final)
        c = eng.bond_curve(hw.Rng(31338, n))
        steps = np.linspace(3, ns - 3, 100).round().astype(int)
        caps = schedule(hw, steps, Tf / ns, Tf, c["P"], tau=0.25)
        assert len(caps) == 100 and len(np.unique(steps)) == 100
        got = eng.cap_floor(hw.Rng(6, n).seek(1), caps, c["P"], c["f"], kind="floor")
        ref = cap_oracle.cap_moments(o, 6, n, caps, c["P"], c["f"], kind="floor", offset=1)
        check(got, ref, rel=5e-6, what="100 caplets")
    finally:
        eng.close()


# ---------------------------------------------------------------- 4. degenerate caplets and the host algebra
def degenerate(hw, P):
    caps = np.concatenate([
        schedule(hw, [200], 0.01, 10.0, P, tau=1.0),        # K far below every P: a caplet that never pays
        schedule(hw, [300], 0.01, 10.0, P, tau=1.0),        # K above every P: always pays
        schedule(hw, [500], 0.01, 10.0, P, tau=0.5),        # at the money
        schedule(hw, [900], 0.01, 10.0, P, tau=1.0),        # T_pay == T_final: interp_mkt's end branch
    ])
    caps["K"][0], caps["K"][1] = 0.01, 2.0
    assert caps["T_pay"][3] == np.float32(10.0)
    return caps


def algebra(mom, n_pairs, control_mean):
    """hw1f_cap_result from five pair moments (include/hw1f.h: n_pairs samples of the pair means X/2, Y/2)"""
    n = float(n_pairs)
    sx, sy, sxx, syy, sxy = 0.5 * mom[0], 0.5 * mom[1], 0.25 * mom[2], 0.25 * mom[3], 0.25 * mom[4]
    mx, my = sx / n, sy / n
    d = n - 1.0 if n > 1.0 else 1.0
    vxx, vyy, cxy = max((sxx - sx * mx) / d, 0.0), max((syy - sy * my) / d, 0.0), (sxy - sx * my) / d
    beta = cxy / vyy if vyy > 0 else 0.0
    vcv = max(vxx - 2 * beta * cxy + beta * beta * vyy, 0.0)
    return dict(price_raw=mx, se_raw=np.sqrt(vxx / n), beta=beta, price_cv=mx - beta * (my - control_mean),
                se_cv=np.sqrt(vcv / n), corr=(cxy / np.sqrt(vxx * vyy) if vxx > 0 and vyy > 0 else 0.0),
                control_mean=control_mean)


STATS = ("price_raw", "se_raw", "beta", "price_cv", "se_cv", "corr", "control_mean")


def test_degenerate_caplets_and_algebra(engine, hw, oracle, curve):
    P, f = curve["P"], curve["f"]
    caps = degenerate(hw, P)
    got = engine.cap_floor(hw.Rng(SEED + 3, N).seek(2), caps, P, f, kind="cap")
    for k in STATS:
        assert np.isfinite(got[k]).all() and np.isfinite(got["strip"][k]), k
    for k in ("price_raw", "price_cv", "se_raw", "se_cv", "beta", "corr"):
        assert got[k][0] == 0.0, k                          # X == 0 on every path: no 0/0
    assert (got["mom"][0][[0, 2, 4]] == 0).all()
    assert got["price_raw"][1] > 0 and got["se_raw"][1] > 0
    ref = cap_oracle.cap_moments(oracle, SEED + 3, N, caps, P, f, kind="cap", offset=2)
    check(got, ref, what="degenerate strip")
    # the host algebra, recomputed in float64 from the returned moments and P_mkt
    means = [float(c["N"]) * interp_mkt(P, float(c["T_pay"]), 10.0, len(P)) for c in caps]
    assert means[3] == float(caps["N"][3]) * float(P[-1])
    rows = [algebra(got["mom"][i], N, means[i]) for i in range(len(caps))]
    rows.append(algebra(np.asarray(got["strip"]["mom"]), N, sum(means)))
    for i, want in enumerate(rows):
        have = got["strip"] if i == len(caps) else {k: got[k][i] for k in STATS}
        for k in STATS:
            assert have[k] == pytest.approx(want[k], rel=1e-12, abs=1e-300), (i, k, have[k], want[k])


def test_finish_beyond_int_range(engine, hw, curve):
    """moments of 2^13 pairs scaled by 2^19 stand in for a 2^32-subsequence run: prices are unchanged, standard
    errors shrink by sqrt(((n - 1) / (n S - 1)) ~ 1 / sqrt(S)"""
    import torch
    SCALE = 1 << 19
    P, f = curve["P"], curve["f"]
    caps = schedule(hw, SEG_STEPS, 0.01, 10.0, P)
    nq = 5 * (len(caps) + 1)
    mom = torch.zeros(nq, dtype=torch.float64, device="cuda")
    torch.cuda.synchronize()
    engine.cap_floor_moments(hw.Rng(SEED + 4, N), caps, P, f, mom.data_ptr(), kind="floor")
    engine.synchronize()
    small = engine.cap_floor_finish(mom.data_ptr(), N, caps, P)
    big_mom = mom * float(SCALE)
    torch.cuda.synchronize()
    assert N * SCALE >= 1 << 32
    big = engine.cap_floor_finish(big_mom.data_ptr(), N * SCALE, caps, P)
    shrink = np.sqrt((N - 1.0) / (N * SCALE - 1.0))
    for a, b in ((small, big), (small["strip"], big["strip"])):
        for k in ("price_raw", "price_cv", "beta", "corr", "control_mean"):
            assert np.allclose(b[k], a[k], rtol=1e-12, atol=0), k
        for k in ("se_raw", "se_cv"):
            assert np.allclose(b[k], np.asarray(a[k]) * shrink, rtol=1e-12, atol=0), k
            assert np.allclose(b[k], np.asarray(a[k]) / np.sqrt(SCALE), rtol=1e-3, atol=0), k


# ---------------------------------------------------------------- 5. state across calls
def test_set_model_round_trip(engine, hw, curve):
    """the noise-free tables the strip uploads (det_m / det_I at the reset steps) follow the engine's model"""
    P, f = curve["P"], curve["f"]
    caps = schedule(hw, SEG_STEPS, 0.01, 10.0, P)
    other = dict(n_steps=500, n_mat=101, r0=0.03)
    e = hw.Engine(device=0)
    e.set_mode(engine.mode)
    try:
        first = e.cap_floor(hw.Rng(SEED + 5, N + 77).seek(1), caps, P, f, kind="cap")
        e.set_model(hw.default_params(**other))
        c2 = e.bond_curve(hw.Rng(SEED, N))
        caps2 = schedule(hw, [5, 100, 250, 399], 0.02, 10.0, c2["P"])
        mid = e.cap_floor(hw.Rng(SEED + 6, N), caps2, c2["P"], c2["f"], kind="floor")
        e.set_model(hw.default_params())
        again = e.cap_floor(hw.Rng(SEED + 5, N + 77).seek(1), caps, P, f, kind="cap")
    finally:
        e.close()
    assert np.array_equal(first["mom"], again["mom"]) and first["strip"] == again["strip"]
    fresh = hw.Engine(device=0, params=hw.default_params(**other))
    fresh.set_mode(engine.mode)
    try:
        want = fresh.cap_floor(hw.Rng(SEED + 6, N), caps2, c2["P"], c2["f"], kind="floor")
    finally:
        fresh.close()
    assert np.array_equal(mid["mom"], want["mom"]) and mid["strip"] == want["strip"]
