"""Caps and floors on the CPU: the strip oracle (tests/cap_oracle.c, the reference-order float sequence evaluated
at every reset step) against the Hull-White closed form, and the rate-to-bond conversion of caplet_schedule."""
import numpy as np
import pytest

import cap_oracle
from cap_closed_form import atm_rate, continuous_theta, interp_mkt, pair_algebra, strip_closed_form

N_CURVE = 1 << 16
N_CAP = 1 << 13


def test_caplet_schedule_rate_to_bond(hw):
    resets = np.array([0.25, 0.5, 1.0])
    pays = np.array([0.5, 1.0, 2.0])
    kappa, M = 0.031, 250.0
    s = hw.caplet_schedule(resets, pays, kappa, notional=M)
    tau = pays - resets
    assert s.dtype.itemsize == 24 and (s["n_steps_reset"] == -1).all()
    np.testing.assert_allclose(s["K"], 1.0 / (1.0 + tau * kappa), rtol=1e-7)
    np.testing.assert_allclose(s["N"], M * (1.0 + tau * kappa), rtol=1e-7)
    # the caplet M tau (L - kappa)^+ paid at T_p, seen at T_r where the bond is P, is N (K - P)^+ with L = (1/P - 1)/tau
    for P in (0.93, 0.97, 0.99, 0.999):
        L = (1.0 / P - 1.0) / tau
        caplet = P * M * tau * np.maximum(L - kappa, 0.0)
        floorlet = P * M * tau * np.maximum(kappa - L, 0.0)
        bond = s["N"].astype(np.float64)
        np.testing.assert_allclose(caplet, bond * np.maximum(s["K"] - P, 0.0), rtol=0, atol=2e-7 * M)   # K, N are float32
        np.testing.assert_allclose(floorlet, bond * np.maximum(P - s["K"], 0.0), rtol=0, atol=2e-7 * M)   # K, N are float32
    per = hw.caplet_schedule(resets, pays, [0.01, 0.02, 0.03], notional=[1.0, 2.0, 3.0])
    np.testing.assert_allclose(per["N"], [1.0 * 1.0025, 2.0 * 1.01, 3.0 * 1.03], rtol=1e-7)
    with pytest.raises(ValueError):
        hw.caplet_schedule([0.5], [1.0, 2.0], 0.02)


@pytest.fixture(scope="module")
def model():
    from oracle_lib import Oracle
    o = Oracle(**continuous_theta())
    s, q = o.bond_curve_sums(777, N_CURVE)
    P, f = o.curve_finalize(s, N_CURVE)
    n = float(N_CURVE)
    x, xx = 0.5 * s, 0.25 * q
    P_se = np.sqrt(np.maximum((xx - x * x / n) / (n - 1), 0.0) / n).astype(np.float32)
    P_se[0] = 0.0
    return o, P, f, P_se


@pytest.mark.parametrize("kind", ["cap", "floor"])
def test_oracle_strip_vs_closed_form(hw, model, kind):
    o, P, f, P_se = model
    Tf, a, sigma = float(o.p.T_final), float(o.p.a), float(o.p.sigma)
    resets = 0.25 * np.arange(1, 40)
    pays = resets + 0.25
    kappa = atm_rate(P, resets, pays, Tf)
    caps = hw.caplet_schedule(resets, pays, kappa)
    mom = cap_oracle.cap_moments(o, 4242, N_CAP, caps, P, f, kind=kind)
    cf, cf_strip = strip_closed_form(kind, caps, P, a, sigma, Tf)
    up, _ = strip_closed_form(kind, caps, P + P_se, a, sigma, Tf)
    dn, _ = strip_closed_form(kind, caps, P - P_se, a, sigma, Tf)
    allow = np.abs(up - dn)
    n_mat = len(P)
    cm = np.array([float(c["N"]) * interp_mkt(P, c["T_pay"], Tf, n_mat) for c in caps])
    for i in range(len(caps)):
        r = pair_algebra(mom[i], N_CAP, cm[i])
        assert abs(r["price_cv"] - cf[i]) <= 5 * r["se_cv"] + allow[i], (i, r, cf[i], allow[i])
    r = pair_algebra(mom[-1], N_CAP, cm.sum())
    assert abs(r["price_cv"] - cf_strip) <= 5 * r["se_cv"] + allow.sum(), (r, cf_strip)
    # the strip's sums are the sums over its caplets
    assert mom[-1][0] == pytest.approx(mom[:-1, 0].sum(), rel=1e-12)
    assert mom[-1][1] == pytest.approx(mom[:-1, 1].sum(), rel=1e-12)
