"""Caps and floors on the GPU (hw1f_cap_floor*): every caplet of a strip in one simulation pass, in both arithmetic modes,
against the CPU oracle, the existing ZBC estimator, the Hull-White closed form and its own standard errors."""
import numpy as np
import pytest

import cap_oracle
from cap_closed_form import atm_rate, continuous_theta, interp_mkt, strip_closed_form

pytestmark = pytest.mark.gpu

N = 1 << 13
SEED = 1234


@pytest.fixture(scope="module")
def curve(engine, hw):
    return engine.bond_curve(hw.Rng(SEED, N))


def quarterly(hw, P, T_final=10.0):
    resets = 0.25 * np.arange(1, 40)            # reset steps 25, 50, ..., 975: odd ones included
    pays = resets + 0.25
    return hw.caplet_schedule(resets, pays, atm_rate(P, resets, pays, T_final))


def one(T_reset, T_pay, K, N_, step=-1):
    return np.array([(T_reset, T_pay, K, N_, step, 0)],
                    dtype=[("T_reset", "f4"), ("T_pay", "f4"), ("K", "f4"), ("N", "f4"), ("n_steps_reset", "i4"),
                           ("reserved", "i4")])


def all_moments(res):
    return np.vstack([res["mom"], np.asarray(res["strip"]["mom"])[None, :]])


@pytest.mark.parametrize("kind", ["cap", "floor"])
@pytest.mark.parametrize("offset", [0, 499])
def test_cap_moments_vs_oracle(engine, hw, oracle, curve, kind, offset):
    caps = quarterly(hw, curve["P"])
    rng = hw.Rng(SEED + 99, N).seek(offset)
    got = engine.cap_floor(rng, caps, curve["P"], curve["f"], kind=kind)
    assert rng.tell() == offset + 975
    ref = cap_oracle.cap_moments(oracle, SEED + 99, N, caps, curve["P"], curve["f"], kind=kind, offset=offset)
    mom = all_moments(got)
    # The bound of test_zbc_moments_vs_oracle (3e-6 relative), plus what MUFU.EX2 (the engine) vs exp2f (the oracle) may
    # leave in the payoff: P = A ex2(..) differs by up to EPS relative, and x = D (K - P)^+ inherits that error in ABSOLUTE
    # terms, |dx| <= EPS y.  Near the money a quarterly caplet's K - P is ~1 % of P, so relative to the payoff the
    # difference is amplified ~100x (the few-step ZBC cases of that test are the same effect); the controls are not.
    EPS = 2.4e-7
    sX, sY, sXX, sYY, sXY = ref.T
    slack = np.stack([EPS * sY, 0 * sY, 2 * EPS * sXY, 0 * sY, EPS * sYY], axis=1)
    gap = np.abs(mom - ref)
    rel = gap / ref
    print(f"{kind} offset {offset}: worst relative moment gap vs oracle {rel.max():.3g} (controls {rel[:, [1, 3]].max():.3g}), "
          f"worst gap / bound {(gap / (3e-6 * ref + slack)).max():.3g}")
    assert (gap <= 3e-6 * ref + slack).all(), (rel.max(), np.unravel_index(rel.argmax(), rel.shape))


def test_one_floorlet_is_the_zbc(engine, hw, curve):
    K = engine.K_DEFAULT
    r1, r2 = hw.Rng(SEED + 7, N), hw.Rng(SEED + 7, N)
    z = engine.zbc_cv(r1, curve["P"], curve["f"], S1=5.0, S2=10.0, K=K, n_steps_S1=500)
    c = engine.cap_floor(r2, one(5.0, 10.0, K, 1.0, 500), curve["P"], curve["f"], kind="floor")
    assert r1.tell() == r2.tell() == 500
    gap = [abs(c["mom"][0][k] / z["mom"][k] - 1) for k in (0, 1)]
    print(f"floorlet vs ZBC: relative gap of sum X {gap[0]:.3g}, of sum Y {gap[1]:.3g}")
    assert max(gap) <= 1e-6, gap
    assert c["price_raw"][0] == pytest.approx(z["mom"][0] / (2 * N), rel=1e-6)
    assert c["strip"]["mom"][0] == pytest.approx(c["mom"][0][0], rel=1e-6)


@pytest.fixture(scope="module")
def cf_setup(engine, hw):
    eng = hw.Engine(device=0, params=hw.default_params(**continuous_theta()))
    eng.set_mode(engine.mode)
    c = eng.bond_curve(hw.Rng(20251, 1 << 21))
    yield eng, c
    eng.close()


def test_strip_vs_closed_form(cf_setup, hw):
    eng, c = cf_setup
    P, f, P_se = c["P"], c["f"], c["P_se"]
    p = eng.params
    resets = 0.5 * np.arange(1, 20)
    pays = resets + 0.5
    caps = hw.caplet_schedule(resets, pays, atm_rate(P, resets, pays, p.T_final))
    got = {}
    for seed, kind in ((31, "cap"), (32, "floor")):
        got[kind] = g = eng.cap_floor(hw.Rng(seed, 1 << 20), caps, P, f, kind=kind)
        cf, cf_strip = strip_closed_form(kind, caps, P, p.a, p.sigma, p.T_final)
        up, _ = strip_closed_form(kind, caps, P + P_se, p.a, p.sigma, p.T_final)
        dn, _ = strip_closed_form(kind, caps, P - P_se, p.a, p.sigma, p.T_final)
        allow = np.abs(up - dn)
        dev = np.abs(g["price_cv"] - cf)
        assert (dev <= 4 * g["se_cv"] + allow).all(), (kind, dev / g["se_cv"], allow)
        assert abs(g["strip"]["price_cv"] - cf_strip) <= 4 * g["strip"]["se_cv"] + allow.sum(), (kind, g["strip"], cf_strip)
        assert g["strip"]["price_raw"] == pytest.approx(g["price_raw"].sum(), rel=1e-6)
    # cap - floor = payer swap: sum N (K P0(T_r) - P0(T_p))
    n = len(P)

    def swap(curve_):
        return sum(float(cp["N"]) * (float(cp["K"]) * interp_mkt(curve_, cp["T_reset"], p.T_final, n)
                                     - interp_mkt(curve_, cp["T_pay"], p.T_final, n)) for cp in caps)

    diff = got["cap"]["strip"]["price_cv"] - got["floor"]["strip"]["price_cv"]
    se = np.hypot(got["cap"]["strip"]["se_cv"], got["floor"]["strip"]["se_cv"])
    assert abs(diff - swap(P)) <= 4 * se + abs(swap(P + P_se) - swap(P - P_se)), (diff, swap(P), se)


@pytest.mark.parametrize("kind", ["cap", "floor"])
def test_standard_errors_are_honest(engine, hw, curve, kind):
    caps = quarterly(hw, curve["P"])
    seeds = [700001 + 7919 * k for k in range(40)]
    runs = [engine.cap_floor(hw.Rng(s, 1 << 16), caps, curve["P"], curve["f"], kind=kind) for s in seeds]
    for est, se in (("price_cv", "se_cv"), ("price_raw", "se_raw")):
        strip = np.array([r["strip"][est] for r in runs])
        ratio = np.mean([r["strip"][se] for r in runs]) / strip.std(ddof=1)
        assert 0.75 < ratio < 1.25, (est, ratio)
        x = np.array([r[est] for r in runs])
        rc = np.array([r[se] for r in runs]).mean(axis=0) / x.std(axis=0, ddof=1)
        assert 0.75 < np.median(rc) < 1.25, (est, np.median(rc))
        assert rc.min() > 0.55 and rc.max() < 1.6, (est, rc.min(), rc.max())


def test_split_form(engine, hw, curve):
    import torch
    caps = quarterly(hw, curve["P"])
    nq = 5 * (len(caps) + 1)
    full = torch.zeros(nq, dtype=torch.float64, device="cuda")
    a_part, b_part = torch.zeros_like(full), torch.zeros_like(full)
    a = 3 * 1024 + 17
    rng = hw.Rng(SEED + 5, N).seek(3)
    engine.cap_floor_moments(rng, caps, curve["P"], curve["f"], full.data_ptr(), kind="cap")
    assert rng.tell() == 3 + 975
    engine.cap_floor_moments(hw.Rng(SEED + 5, a).seek(3), caps, curve["P"], curve["f"], a_part.data_ptr(), kind="cap")
    engine.cap_floor_moments(hw.Rng(SEED + 5, N - a, first_path=a).seek(3), caps, curve["P"], curve["f"],
                             b_part.data_ptr(), kind="cap")
    engine.synchronize()
    f_, s_ = full.cpu().numpy(), (a_part + b_part).cpu().numpy()
    assert np.allclose(f_, s_, rtol=2e-6, atol=0), np.abs(f_ / s_ - 1).max()
    fin = engine.cap_floor_finish(full.data_ptr(), N, caps, curve["P"])
    one_call = engine.cap_floor(hw.Rng(SEED + 5, N).seek(3), caps, curve["P"], curve["f"], kind="cap")
    for k in ("price_cv", "se_cv", "price_raw", "se_raw", "beta", "corr", "control_mean", "mom"):
        assert np.array_equal(fin[k], one_call[k]), k
    assert fin["strip"] == one_call["strip"]


def test_bit_reproducible(engine, hw, curve):
    caps = quarterly(hw, curve["P"])
    r = [engine.cap_floor(hw.Rng(SEED + 3, N + 333).seek(1), caps, curve["P"], curve["f"], kind="floor") for _ in range(2)]
    assert np.array_equal(r[0]["mom"], r[1]["mom"]) and r[0]["strip"] == r[1]["strip"]
    assert np.array_equal(r[0]["price_cv"], r[1]["price_cv"])


def test_rejected_arguments(engine, hw, curve):
    P, f = curve["P"], curve["f"]
    Tf, n_steps = float(engine.params.T_final), engine.n_steps
    good = one(1.0, 2.0, 0.98, 1.0)
    two = np.concatenate([one(0.5, 1.0, 0.98, 1.0), one(0.25, 1.0, 0.98, 1.0)])
    cases = [
        ("kind", good, 2),
        ("n_caplets 0", good[:0], "cap"),
        ("n_caplets 101", np.repeat(good, 101), "cap"),
        ("decreasing steps", two, "cap"),
        ("step 0", one(1.0, 2.0, 0.98, 1.0, 0), "cap"),
        ("step beyond n_steps", one(1.0, 2.0, 0.98, 1.0, n_steps + 1), "cap"),
        ("T_pay == T_reset", one(1.0, 1.0, 0.98, 1.0), "floor"),
        ("T_pay > T_final", one(1.0, Tf + 0.5, 0.98, 1.0), "cap"),
        ("T_reset off the grid", one(1.0037, 2.0, 0.98, 1.0), "cap"),
        ("K = 0", one(1.0, 2.0, 0.0, 1.0), "cap"),
        ("K = nan", one(1.0, 2.0, np.nan, 1.0), "cap"),
        ("N < 0", one(1.0, 2.0, 0.98, -1.0), "cap"),
        ("N = inf", one(1.0, 2.0, 0.98, np.inf), "floor"),
    ]
    for name, caps, kind in cases:
        rng = hw.Rng(SEED, N).seek(7)
        before = engine.launch_count
        with pytest.raises(hw.HW1FError) as ei:
            engine.cap_floor(rng, caps, P, f, kind=kind)
        assert ei.value.status == hw._ffi.ERR_INVALID, name
        assert len(str(ei.value).split(":", 1)[1].strip()) > 10, (name, str(ei.value))
        with pytest.raises(hw.HW1FError):
            engine.cap_floor_moments(rng, caps, P, f, 0, kind=kind)
        assert engine.launch_count == before, name
        assert rng.tell() == 7, name
